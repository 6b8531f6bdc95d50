"""Host-side mirror of the reference's engine interface for the accelerated path.

Same class names, constructor arguments and call signatures as gat/Engine.pyx so that gat-run.py-style
code and the reference's own tests read the same:

    containers   IntervalDictionary (Engine.pyx:2741-2880), IntervalCollection (:2887-3165)
    sampler      SamplerAnnotator(bucket_size, nbuckets).sample(segments, workspace)   (:445-646)
    counters     Counter*()(segments, annotations, workspace) and .name                 (:1412-1472)
    workspace    UnconditionalWorkspace                                                  (:2061-2069)
    counts       computeCounts(...)                                                      (:2164-2204)
    results      AnnotatorResult / AnnotatorResultExtended                               (:1725-1974)
    p/q values   updatePValues, getQValues, updateQValues                                (:1976-2054)

The objects hold no algorithm: SamplerAnnotator.sample, Counter.__call__, computeCounts and the result
statistics all execute in libgat_b200.so on the GPU (gat_b200/device.py); there is no CPU fallback.
"""
import collections
import math
import os

import numpy as np

from . import device as _dev
from . import stats as Stats
from .segmentlist import SegmentList

# --------------------------------------------------------------------------------------- GPU context
_context = {}


def getContext(device=None):
    """the process-wide gat_b200 Context of a GPU (default: LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _context:
        _context[device] = _dev.Context(device)
    return _context[device]


_rng_state = {"seed": None, "calls": 0}


def seed(value):
    """seed the placement stream (counterpart of numpy.random.seed in scripts/gat-run.py:267-271)."""
    _rng_state["seed"] = int(value) & 0xFFFFFFFFFFFFFFFF
    _rng_state["calls"] = 0


def getSeed():
    if _rng_state["seed"] is None:
        # like the reference, an unseeded run draws its seed from numpy's global generator
        seed(int(np.random.randint(0, 2 ** 31 - 1)))
    return _rng_state["seed"]


# --------------------------------------------------------------------------------------- containers
class IntervalContainer(object):
    """generic collection of SegmentLists (gat/Engine.pyx:2559-2738); share()/unshare() exist for API
    compatibility only -- there is no multiprocessing on this path."""

    def __init__(self):
        self.name = None

    def getName(self):
        return self.name

    def setName(self, name):
        self.name = name

    def share(self, filename=None):
        pass

    def unshare(self):
        pass

    def sum(self):
        # one vectorised pass over all lists (a Python-level sum of per-list sums costs ~5 us per list, and
        # gat.run asks for the size of every annotation)
        arrays = [s.asarray() for s in self.getSegmentLists() if len(s)]
        if not arrays:
            return 0
        a = arrays[0] if len(arrays) == 1 else np.concatenate(arrays, axis=0)
        return int(a[:, 1].sum(dtype=np.int64)) - int(a[:, 0].sum(dtype=np.int64))

    def counts(self):
        return sum(len(s) for s in self.getSegmentLists())

    def sort(self):
        for s in self.getSegmentLists():
            s.sort()

    def normalize(self):
        for s in self.getSegmentLists():
            s.normalize()

    def check(self):
        self.sort()


class IntervalDictionary(IntervalContainer):
    """key (contig or contig.isochore) -> SegmentList (gat/Engine.pyx:2741-2880)."""

    def __init__(self, name=None):
        IntervalContainer.__init__(self)
        self.intervals = collections.defaultdict(SegmentList)
        self.name = name

    def getSegmentLists(self):
        for _, s in list(self.intervals.items()):
            yield s

    def __len__(self):
        return len(self.intervals)

    def __str__(self):
        return ";".join("%s:%i,%i" % (x, len(y), y.sum()) for x, y in self.intervals.items())

    def __delitem__(self, key):
        del self.intervals[key]

    def __getitem__(self, key):
        return self.intervals[key]

    def __setitem__(self, key, val):
        self.intervals[key] = val

    def __contains__(self, key):
        return key in self.intervals

    def keys(self):
        return self.intervals.keys()

    def items(self):
        return self.intervals.items()

    def add(self, contig, segmentlist):
        self.intervals[contig] = segmentlist

    def clone(self):
        r = IntervalDictionary()
        for contig, s in self.intervals.items():
            r[contig] = s.clone()
        return r

    def _apply(self, other, op):
        drop = []
        for contig, s in self.intervals.items():
            if contig in other:
                getattr(s, op)(other[contig])
            else:
                drop.append(contig)
        for contig in drop:
            del self.intervals[contig]

    def filter(self, other):
        """keep intervals overlapping intervals in other; contigs absent from other vanish"""
        self._apply(other, "filter")

    def intersect(self, other):
        self._apply(other, "intersect")

    def toIsochores(self, isochores, truncate=False, _pieces=None):
        """split key `contig` into `contig.isochore` per isochore track (gat/Engine.pyx:2837-2855)"""
        for contig in list(self.intervals.keys()):
            s = self.intervals[contig]
            if not (truncate and self._truncate_all(contig, s, isochores, _pieces)):
                for iso_track, iso in isochores.items():
                    n = s.clone()
                    if truncate:
                        n.intersect(iso[contig])
                    else:
                        n.filter(iso[contig])
                    self.intervals["%s.%s" % (contig, iso_track)] = n
            del self.intervals[contig]

    def _truncate_all(self, contig, s, isochores, cache=None):
        """`s.clone().intersect(iso[contig])` for every isochore track in ONE pass: the pieces of all tracks on
        the contig form one sorted disjoint list when the isochores do not overlap each other (the usual case: they
        partition the genome), so a single pair of searches gives every (segment, piece) pair and the piece's track
        says where the truncated segment goes.  Same lists, same order as the per-track loop; returns False
        (nothing done) when the isochore tracks overlap or a list is not normalized."""
        if cache is not None and contig in cache:          # (the same isochores for every track of a collection)
            tracks, pieces, label = cache[contig]
        else:
            tracks = [(t, iso[contig]) for t, iso in isochores.items()]
            pieces = label = None
            arrs = [p.asarray() for _, p in tracks]
            if all(p.isNormalized for _, p in tracks) and sum(len(a) for a in arrs) > 0:
                pieces = np.concatenate(arrs)
                label = np.repeat(np.arange(len(arrs)), [len(a) for a in arrs])
                order = np.argsort(pieces[:, 0], kind="stable")
                pieces, label = pieces[order], label[order]
                if len(pieces) > 1 and (pieces[1:, 0] < pieces[:-1, 1]).any():
                    pieces = label = None
            if cache is not None:
                cache[contig] = (tracks, pieces, label)
        if pieces is None or len(s) == 0 or not s.isNormalized:
            return False
        a = s.asarray()
        j1 = np.searchsorted(pieces[:, 1], a[:, 0], side="right")       # first piece ending after the start
        j2 = np.maximum(j1, np.searchsorted(pieces[:, 0], a[:, 1], side="left"))
        cnt = j2 - j1
        total = int(cnt.sum())
        rep = np.repeat(np.arange(len(a)), cnt)
        pj = np.repeat(j1, cnt) + (np.arange(total) - np.repeat(np.cumsum(cnt) - cnt, cnt))
        out = np.empty((total, 2), dtype=np.uint32)
        out[:, 0] = np.maximum(a[rep, 0], pieces[pj, 0])
        out[:, 1] = np.minimum(a[rep, 1], pieces[pj, 1])
        where = label[pj]
        for i, (t, _) in enumerate(tracks):
            n = SegmentList(array=out[where == i])
            n._normalized = True
            self.intervals["%s.%s" % (contig, t)] = n
        return True

    def fromIsochores(self):
        """merge `contig.isochore` keys back into contigs; merge(0) when any key was split
        (gat/Engine.pyx:2857-2876)"""
        new = collections.defaultdict(SegmentList)
        normalize = False
        for isochore, s in self.intervals.items():
            isochore = isochore.strip()
            if "." in isochore and isochore != ".":
                contig, _ = isochore.split(".")
                new[contig].extend(s)
                normalize = True
            else:
                new[isochore] = s
        if normalize:
            for x in new.values():
                x.merge(0)
        self.intervals = new


class IntervalCollection(IntervalContainer):
    """track -> IntervalDictionary (gat/Engine.pyx:2887-3165)."""

    def __init__(self, name=None):
        IntervalContainer.__init__(self)
        self.intervals = collections.defaultdict(IntervalDictionary)
        self.name = name

    def getSegmentLists(self):
        for _, v in list(self.intervals.items()):
            for _, s in list(v.items()):
                yield s

    def load(self, filenames, allow_multiple=False, ignore_tracks=False):
        from .io import readFromBed
        self.intervals = readFromBed(filenames, allow_multiple=allow_multiple, ignore_tracks=ignore_tracks)

    def save(self, outfile, prefix="", **kwargs):
        for track, vv in self.intervals.items():
            outfile.write("track name=%s%s %s\n" % (prefix, track, " ".join("%s=%s" % kv for kv in kwargs.items())))
            for contig, s in vv.items():
                for start, end in s:
                    outfile.write("%s\t%i\t%i\n" % (contig, start, end))

    def normalize(self):
        """normalize every list; contigs without segments are removed (gat/Engine.pyx:2941-2956)"""
        for track, vv in self.intervals.items():
            for contig in [c for c in vv.keys() if len(vv[c]) == 0]:
                del vv[contig]
            for contig in vv.keys():
                vv[contig].normalize()

    def merge(self, delete=False):
        """pool all tracks into track 'merged' (not normalized)"""
        merged = IntervalDictionary()
        for track in list(self.intervals.keys()):
            for contig, s in self.intervals[track].items():
                merged[contig].extend(s)
            if delete:
                del self.intervals[track]
        self.intervals["merged"] = merged

    def collapse(self):
        """track 'collapsed' = intersection of all tracks on the contigs they share"""
        ntracks = len(self.intervals)
        seen = collections.Counter(c for vv in self.intervals.values() for c in vv.keys())
        shared = set(c for c, n in seen.items() if n == ntracks)
        result = IntervalDictionary()
        for track, vv in self.intervals.items():
            for contig, s in vv.items():
                if contig not in shared:
                    continue
                if contig not in result:
                    result[contig] = s.clone()
                else:
                    result[contig].intersect(s)
        self.intervals["collapsed"] = result

    def countsPerTrack(self):
        return dict((track, sum(len(s) for _, s in vv.items())) for track, vv in self.intervals.items())

    def intersect(self, other):
        for vv in self.intervals.values():
            vv.intersect(other)

    def filter(self, other):
        for vv in self.intervals.values():
            vv.filter(other)

    def restrict(self, restrict):
        keep = set(restrict) if isinstance(restrict, (list, tuple, set)) else set([restrict])
        for track in [t for t in self.intervals.keys() if t not in keep]:
            del self.intervals[track]

    def toIsochores(self, isochores, truncate=False):
        pieces = {}             # per contig: the isochore pieces of all tracks as one sorted list (shared by the tracks)
        for vv in self.intervals.values():
            vv.toIsochores(isochores, truncate, pieces)

    def fromIsochores(self):
        for vv in self.intervals.values():
            vv.fromIsochores()

    def clone(self):
        new = IntervalCollection(self.name)
        for track, v in self.intervals.items():
            for contig, s in v.items():
                new.add(track, contig, s.clone())
        return new

    @property
    def tracks(self):
        return self.intervals.keys()

    def __len__(self):
        return len(self.intervals)

    def __delitem__(self, key):
        del self.intervals[key]

    def __getitem__(self, key):
        return self.intervals[key]

    def __contains__(self, key):
        return key in self.intervals

    def keys(self):
        return self.intervals.keys()

    def items(self):
        return self.intervals.items()

    def add(self, track, contig, segmentlist):
        self.intervals[track][contig] = segmentlist

    def __str__(self):
        return "%s:%s" % (self.name, ",".join("%s:%s" % (x, y) for x, y in self.intervals.items()))

    def outputStats(self, outfile):
        outfile.write("section\ttrack\tcontig\tnsegments\tlength\n")
        for track, vv in self.intervals.items():
            tl = ts = 0
            for contig, s in vv.items():
                outfile.write("\t".join((str(self.name), track, contig, "%i" % len(s), "%i" % s.sum())) + "\n")
                tl += s.sum()
                ts += len(s)
            outfile.write("\t".join((str(self.name), track, "total", "%i" % ts, "%i" % tl)) + "\n")


class DeviceIntervalCollection(IntervalCollection):
    """An IntervalCollection whose lists live on the GPU (device.Lists, CSR: list = track x key) -- the large
    annotation collection between BED parsing and the index build (SURVEY 8 f1).  normalize / intersect / filter /
    toIsochores / fromIsochores / clone / sum / counts run as a few device passes over ALL lists at once instead of
    one numpy call per (track, contig) list (24 000 of them at 1000 tracks), and gat_b200.run builds the annotation
    index from the device lists without the intervals returning to the host.

    Reading through the dictionary interface (`coll[track][contig]`, items(), save ...) hands out a host SNAPSHOT of
    the lists; structural changes that this class does not implement on the device (add, merge, collapse, restrict,
    deleting tracks) turn it into an ordinary host collection (same results, host speed).  Same semantics as the
    reference's container: gat/Engine.pyx:2887-3165, gat/IO.py:188-293."""

    def __init__(self, name=None):
        IntervalContainer.__init__(self)
        self.name = name
        self._tracks = []           # track names, in order of first appearance
        self._keys = []             # keys (contig or contig.isochore), shared by all tracks
        self._exists = None         # bool [tracks][keys]: the key is in the track's dictionary
        self._lists = None          # device.Lists, list t * len(keys) + k
        self._rows = None           # loaded but not yet normalized: (list_id, start, end, grouper)
        self._fanout = 0            # > 0 after toIsochores: keys = contigs x isochore tracks, contig-major
        self._snapshot = None       # host view of the device lists
        self._plain = None          # the host dictionary once the collection has been demoted

    # ---- state -----------------------------------------------------------------------------------------------
    @property
    def onDevice(self):
        return self._plain is None and (self._lists is not None or self._rows is not None)

    @property
    def intervals(self):
        if self._plain is not None:
            return self._plain
        if self._snapshot is None:
            self._snapshot = self._materialize()
        return self._snapshot

    @intervals.setter
    def intervals(self, value):         # (IntervalCollection.load and friends assign the dictionary)
        self._plain = value
        self._drop_device()

    def _drop_device(self):
        if self._lists is not None:
            self._lists.close()
        self._lists = self._rows = self._snapshot = None

    def _demote(self):
        """become an ordinary host collection (for operations without a device implementation)"""
        if self._plain is None:
            snapshot = self.intervals
            self._plain = snapshot
            self._drop_device()

    def _materialize(self):
        out = collections.defaultdict(IntervalDictionary)
        if self._rows is not None:      # not normalized yet: group the raw rows like the host reader does
            for track, contigs in self._rows[3]().items():
                d = IntervalDictionary()
                for contig, parts in contigs.items():
                    data = parts[0] if len(parts) == 1 else np.concatenate(parts)
                    d[contig] = SegmentList(array=data.astype(np.int64).astype(np.uint32))
                out[track] = d
            return out
        offs, data = self._lists.download()
        K = len(self._keys)
        for t, track in enumerate(self._tracks):
            d = IntervalDictionary()
            for k in np.flatnonzero(self._exists[t]):
                l = t * K + int(k)
                s = SegmentList(array=data[int(offs[l]):int(offs[l + 1])])
                s._normalized = True
                d[self._keys[int(k)]] = s
            out[track] = d
        return out

    def _changed(self, lists):
        if self._lists is not None and lists is not self._lists:
            self._lists.close()
        self._lists = lists
        self._snapshot = None

    # ---- loading ---------------------------------------------------------------------------------------------
    def load(self, filenames, allow_multiple=False, ignore_tracks=False):
        from .io import readFromBed
        flat = readFromBed(filenames, allow_multiple=allow_multiple, ignore_tracks=ignore_tracks, flat=True)
        if "grouper" not in flat:           # a file needed the line-by-line reader: host collection
            self.intervals = flat
            return
        self._plain = None
        self._tracks, self._keys = list(flat["tracks"]), list(flat["contigs"])
        T, K = len(self._tracks), len(self._keys)
        list_id = flat["track"].astype(np.int64) * K + flat["contig"]
        present = np.zeros(T * K, dtype=bool)
        present[list_id] = True
        self._exists = present.reshape(T, K)
        self._rows = (list_id.astype(np.uint32), flat["start"].astype(np.uint32), flat["end"].astype(np.uint32),
                      flat["grouper"])
        self._lists, self._snapshot, self._fanout = None, None, 0

    def _other_lists(self, dictionaries):
        """device lists of `dictionaries[f][key]` for every key of this collection and every f, key-major; None if
        one of them is not normalized (the device kernels assume sorted, disjoint lists)"""
        empty = np.zeros((0, 2), dtype=np.uint32)
        lists = []
        for key in self._keys:
            for d in dictionaries:
                if key in d:
                    s = d[key]
                    if not s.isNormalized:
                        return None
                    lists.append(s.asarray())
                else:
                    lists.append(empty)
        return _dev.Lists.from_lists(getContext(), lists)

    # ---- operations with a device implementation -----------------------------------------------------------------
    def normalize(self):
        if not self.onDevice:
            return IntervalCollection.normalize(self)
        if self._rows is not None:
            list_id, start, end, _ = self._rows
            lists = _dev.Lists.from_rows(getContext(), list_id, start, end, len(self._tracks) * len(self._keys))
            self._rows = None
            self._changed(lists)
        # (device lists are normalized by construction)

    def _restrict(self, other, truncate):
        others = self._other_lists([other])
        if others is None or self._rows is not None:
            self._demote()
            return False
        self._changed(self._lists.restrict(len(self._keys), 1, others, truncate))
        others.close()
        keep = np.array([key in other for key in self._keys], dtype=bool)      # contigs absent from other vanish
        self._exists = self._exists & keep[None, :]
        return True

    def intersect(self, other):
        if not self.onDevice or not self._restrict(other, True):
            IntervalCollection.intersect(self, other)

    def filter(self, other):
        if not self.onDevice or not self._restrict(other, False):
            IntervalCollection.filter(self, other)

    def toIsochores(self, isochores, truncate=False):
        if self.onDevice and self._rows is None and self._fanout == 0:
            names = list(isochores.keys())
            others = self._other_lists([isochores[n] for n in names]) if names else None
            if others is not None:
                F = len(names)
                self._changed(self._lists.restrict(len(self._keys), F, others, truncate))
                others.close()
                self._keys = ["%s.%s" % (contig, n) for contig in self._keys for n in names]
                self._exists = np.repeat(self._exists, F, axis=1)
                self._fanout = F
                return
        if self.onDevice:
            self._demote()
        IntervalCollection.toIsochores(self, isochores, truncate)

    def fromIsochores(self):
        if self.onDevice and self._rows is None:
            if self._fanout == 0 and not any("." in k.strip() and k.strip() != "." for k in self._keys):
                return                      # no key is split: nothing to do (gat/Engine.pyx:2862-2873)
            if self._fanout > 0:
                F = self._fanout
                self._changed(self._lists.collapse(F))
                self._keys = [k.strip().split(".")[0] for k in self._keys[::F]]
                T = len(self._tracks)
                self._exists = self._exists.reshape(T, -1, F).any(axis=2)
                self._fanout = 0
                return
        if self.onDevice:
            self._demote()
        IntervalCollection.fromIsochores(self)

    def clone(self):
        if not self.onDevice or self._rows is not None:
            return IntervalCollection.clone(self)
        new = DeviceIntervalCollection(self.name)
        new._tracks, new._keys = list(self._tracks), list(self._keys)
        new._exists, new._fanout = self._exists.copy(), self._fanout
        new._lists = self._lists.select(np.arange(self._lists.n_lists, dtype=np.uint32))
        return new

    def sum(self):
        if not self.onDevice or self._rows is not None:
            return IntervalCollection.sum(self)
        return int(self._lists.sizes()[1].sum())

    def counts(self):
        if not self.onDevice or self._rows is not None:
            return IntervalCollection.counts(self)
        return int(self._lists.n_intervals)

    def trackSizes(self):
        """{track: (number of segments, bases)} -- what run() asks every annotation track for"""
        if not self.onDevice or self._rows is not None:
            return dict((t, (self.intervals[t].counts(), self.intervals[t].sum())) for t in self.tracks)
        count, bases = self._lists.sizes()
        K = len(self._keys)
        return dict((t, (int(count[i * K:(i + 1) * K].sum()), int(bases[i * K:(i + 1) * K].sum())))
                    for i, t in enumerate(self._tracks))

    def deviceLists(self, keys):
        """device lists [track][key] for the given keys (an unknown key gives empty lists): the caller closes them"""
        index = dict((k, i) for i, k in enumerate(self._keys))
        K, n = len(self._keys), self._lists.n_lists
        col = np.array([index.get(k, -1) for k in keys], dtype=np.int64)
        src = np.arange(len(self._tracks), dtype=np.int64)[:, None] * K + col[None, :]
        src[:, col < 0] = n
        return self._lists.select(src.reshape(-1).astype(np.uint32))

    # ---- reading ---------------------------------------------------------------------------------------------
    @property
    def tracks(self):
        return list(self._tracks) if self.onDevice else self.intervals.keys()

    def keys(self):
        return self.tracks

    def __len__(self):
        return len(self._tracks) if self.onDevice else len(self.intervals)

    def __contains__(self, key):
        return key in self._tracks if self.onDevice else key in self.intervals

    # ---- structural changes: host only ---------------------------------------------------------------------------
    def __delitem__(self, key):
        self._demote()
        IntervalCollection.__delitem__(self, key)

    def add(self, track, contig, segmentlist):
        self._demote()
        IntervalCollection.add(self, track, contig, segmentlist)

    def merge(self, delete=False):
        self._demote()
        IntervalCollection.merge(self, delete)

    def collapse(self):
        self._demote()
        IntervalCollection.collapse(self)

    def restrict(self, restrict):
        self._demote()
        IntervalCollection.restrict(self, restrict)

    def sort(self):
        if not self.onDevice:
            IntervalCollection.sort(self)
        elif self._rows is not None:
            self._demote()
            IntervalCollection.sort(self)


# ------------------------------------------------------------------------------------------ sampler
class Sampler(object):
    pass


def splitKey(key):
    """contig of a workspace key: 'contig.isochore' -> contig (gat/Engine.pyx:2862-2866)"""
    key = key.strip()
    if "." in key and key != ".":
        return key.split(".")[0], True
    return key, False


class SamplerAnnotator(Sampler):
    """the annotator sampling method (gat/Engine.pyx:445-646) on the GPU.

    `sample(segments, workspace)` places ONE unit and returns a SegmentList, like the reference; it is
    meant for tests and scripts.  gat_b200.run() recognises this class and sends the whole track
    (all units x all samples) to the GPU in one batched call instead."""

    accelerated = True
    kind = "annotator"

    def __init__(self, bucket_size=1, nbuckets=100000, nunsuccessful_rounds=0):
        self.bucket_size = bucket_size
        self.nbuckets = nbuckets
        self.nunsuccessful_rounds = nunsuccessful_rounds

    def __reduce__(self):
        return (SamplerAnnotator, (self.bucket_size, self.nbuckets, self.nunsuccessful_rounds))

    def sample(self, segments, workspace):
        assert segments.isNormalized, "segment list is not normalized"
        assert workspace.isNormalized, "workspace is not normalized"
        if len(segments) == 0 or len(workspace) == 0:
            return SegmentList()
        ctx = getContext()
        try:
            smp = _dev.Sampler(ctx, [0], 1, False, [segments.asarray()], [workspace.asarray()],
                               bucket_size=self.bucket_size, nbuckets=self.nbuckets)
        except _dev._lib.GatB200Error as e:
            if e.code == _dev._lib.ERR_TOO_LARGE:
                raise ValueError(str(e))
            raise
        call = _rng_state["calls"]
        _rng_state["calls"] += 1
        placed, status = smp.place(getSeed(), 0xFFFFFF, call, 1)
        self.nunsuccessful_rounds = 20 if (status[0, 0] & _dev.UNIT_HIT_ROUND_CAP) else 0
        smp.close()
        r = SegmentList(array=placed[0][0])
        r._normalized = True
        return r


class SamplerShift(Sampler):
    """shift every segment by a random amount within *radius* (a multiple of its length) or *extension* bases
    around its midpoint, wrapping around the ends of the local workspace (gat/Engine.pyx:998-1111) -- on the
    GPU (`shift_kernel`).  `sample(segments, workspace)` moves ONE unit, like the reference; gat_b200.run()
    sends the whole track to the GPU in one batched call."""

    accelerated = True
    kind = "shift"
    bucket_size = 1         # (the unit preparation is shared with the other samplers; nbuckets = 0 asks for no
    nbuckets = 0            #  length histogram -- the shift never calls getLengthDistribution, so no segment
                            #  is ever "too large" for it, gat/Engine.pyx:1060-1062)

    def __init__(self, radius=2, extension=0):
        self.radius = radius
        self.extension = int(extension)

    def __reduce__(self):
        return (SamplerShift, (self.radius, self.extension))

    def sample(self, segments, workspace):
        assert workspace.isNormalized, "workspace is not normalized"
        if len(segments) == 0 or len(workspace) == 0:
            return SegmentList()
        ctx = getContext()
        smp = _dev.Sampler(ctx, [0], 1, False, [segments.asarray()], [workspace.asarray()],
                           bucket_size=self.bucket_size, nbuckets=self.nbuckets)
        smp.set_shift(self.radius, self.extension)
        call = _rng_state["calls"]
        _rng_state["calls"] += 1
        try:
            placed, status = smp.place(getSeed(), 0xFFFFFF, call, 1)
        except _dev._lib.GatB200Error as e:
            if e.code == _dev._lib.ERR_CAPACITY:
                raise MemoryError("SamplerShift: the moved segments were cut into more pieces than the buffer holds")
            raise
        finally:
            smp.close()
        r = SegmentList(array=placed[0][0])
        r._normalized = True
        return r


class SamplerSegments(Sampler):
    """sample exactly len(segments) segments from the length distribution (gat/Engine.pyx:653-737).  Its
    samples are unsorted and may overlap; like in the reference they only become countable through the
    merge(0) of IntervalDictionary.fromIsochores, so gat_b200.run() accepts it with isochore workspaces."""

    accelerated = True
    kind = "segments"

    def __init__(self, bucket_size=1, nbuckets=100000):
        self.bucket_size = bucket_size
        self.nbuckets = nbuckets

    def __reduce__(self):
        return (SamplerSegments, (self.bucket_size, self.nbuckets))

    def sample(self, segments, workspace):
        """exactly len(working segments) placements, in draw order, unsorted and possibly overlapping -- the list
        the reference returns (gat/Engine.pyx:719-735); only fromIsochores' merge(0) normalizes it"""
        assert workspace.isNormalized, "workspace is not normalized"
        if len(segments) == 0 or len(workspace) == 0:
            return SegmentList()
        ctx = getContext()
        # one unit declared as an isochore key: the unit-level list is then handed back as drawn
        try:
            smp = _dev.Sampler(ctx, [0], 1, True, [segments.asarray()], [workspace.asarray()],
                               bucket_size=self.bucket_size, nbuckets=self.nbuckets)
        except _dev._lib.GatB200Error as e:
            if e.code == _dev._lib.ERR_TOO_LARGE:
                raise ValueError(str(e))
            raise
        smp.set_kind("segments")
        call = _rng_state["calls"]
        _rng_state["calls"] += 1
        try:
            placed, _ = smp.place_units(getSeed(), 0xFFFFFF, call, 1)
        finally:
            smp.close()
        return SegmentList(array=placed[0][0])


# ----------------------------------------------------------------------------------------- counters
class Counter(object):
    """base class: counts between two segment lists (gat/Engine.pyx:1412-1415)."""
    name = None

    def __call__(self, segments, annotations, workspace=None):
        nseg = [len(workspace)] if workspace is not None else [0]
        if self.name == "nucleotide-density" and nseg[0] == 0:
            return 0
        ctx = getContext()
        annos = _dev.Annotations(ctx, [[annotations.asarray()]], key_ws_nseg=nseg)
        out = annos.count_lists([self.name], [[segments.asarray()]])
        annos.close()
        v = out[0, 0, 0]
        return float(v) if self.name == "nucleotide-density" else int(v)


class CounterNucleotideOverlap(Counter):
    name = "nucleotide-overlap"


class CounterNucleotideDensity(Counter):
    name = "nucleotide-density"


class CounterSegmentOverlap(Counter):
    name = "segment-overlap"


class CounterSegmentMidpointOverlap(Counter):
    name = "segment-midoverlap"


class CounterAnnotationOverlap(Counter):
    name = "annotation-overlap"


class CounterAnnotationMidpointOverlap(Counter):
    name = "annotation-midoverlap"


COUNTER_CLASSES = dict((c.name, c) for c in (CounterNucleotideOverlap, CounterNucleotideDensity,
                                             CounterSegmentOverlap, CounterSegmentMidpointOverlap,
                                             CounterAnnotationOverlap, CounterAnnotationMidpointOverlap))


class UnconditionalWorkspace(object):
    """the default, unconditional workspace (gat/Engine.pyx:2061-2069)."""
    is_conditional = False

    def __call__(self, segments, annotations, workspace):
        return segments, annotations, workspace


# ------------------------------------------------------------------------------------ observed counts
def deviceAnnotations(annotations, keys, nseg=None, cache=None, lazy=False):
    """the annotation tracks on `keys` as a device.Annotations set; `cache` (dict keyed by the key tuple) lets
    the observed counts of every counter, the sampling and the overlap columns of one run share ONE upload
    and index build.  -> (set, owned): the caller closes the set iff owned."""
    k = tuple(keys)
    if cache is not None and k in cache:
        return cache[k], False
    if isinstance(annotations, DeviceIntervalCollection) and annotations.onDevice and annotations._rows is None:
        # the lists are on the GPU already: pick the keys, build the index in place
        picked = annotations.deviceLists(keys)
        obj = _dev.Annotations.from_device_lists(getContext(), picked, len(annotations._tracks), len(keys), nseg)
        picked.close()
    else:
        empty = np.zeros((0, 2), dtype=np.uint32)
        lists = [[annotations[a][key].asarray() if key in annotations[a] else empty for key in keys]
                 for a in annotations.tracks]
        obj = _dev.Annotations(getContext(), lists, key_ws_nseg=nseg, lazy=lazy)
    if cache is not None:
        cache[k] = obj
    return obj, cache is None


def computeCounts(counter, aggregator, segments, annotations, workspace, workspace_generator, append=False,
                  annos_cache=None):
    """observed counts of every (track, annotation) pair: aggregator over workspace keys of
    counter(segs[key], annos[key], workspace[key]) (gat/Engine.pyx:2164-2204).  One batched GPU call
    per counter; only the `sum` aggregator of the reference's call site is supported."""
    if aggregator is not sum:
        raise NotImplementedError("gat_b200.computeCounts supports aggregator=sum only")
    if append:
        counts = collections.defaultdict(list)
    else:
        counts = collections.defaultdict(lambda: collections.defaultdict(float))
    keys = list(workspace.keys())
    tracks = list(segments.tracks)
    atracks = list(annotations.tracks)
    if not keys or not tracks or not atracks:
        return counts
    annos, owned = deviceAnnotations(annotations, keys, [len(workspace[k]) for k in keys], annos_cache)
    empty = np.zeros((0, 2), dtype=np.uint32)
    out = annos.count_lists([counter.name], [[segments[t][k].asarray() if k in segments[t] else empty for k in keys]
                                             for t in tracks])
    if owned:
        annos.close()
    is_float = counter.name == "nucleotide-density"
    for ti, track in enumerate(tracks):
        for ai, annotation in enumerate(atracks):
            v = out[0, ti, ai]
            v = float(v) if is_float else int(v)
            if append:
                counts[annotation].append(v)
            else:
                counts[track][annotation] = v
    return counts


def overlapColumns(track_segments, annotations, annos_cache=None):
    """{annotation: (overlap_nsegments, overlap_size)} of one track against every annotation track: the
    counts() and sum() of track_segments.intersect(annotation_segments) that AnnotatorResultExtended reports
    (gat/Engine.pyx:1911-1928), for all annotations in ONE batched GPU call instead of one host intersect
    per result.  For normalized lists the pieces of intersect() are the overlapping (segment, interval)
    pairs and their total length is the nucleotide overlap."""
    atracks = list(annotations.tracks)
    keys = [k for k in track_segments.keys()]
    if not keys or not atracks:
        return dict((a, (0, 0)) for a in atracks)
    annos, owned = deviceAnnotations(annotations, keys, None, annos_cache)
    out = annos.count_lists(["overlap-pieces", "nucleotide-overlap"], [[track_segments[k].asarray() for k in keys]])
    if owned:
        annos.close()
    return dict((a, (int(out[0, 0, i]), int(out[1, 0, i]))) for i, a in enumerate(atracks))


# ------------------------------------------------------------------------------------------- results
class SampleMatrix(object):
    """The S x A matrix of sampled counts of one (track, counter), left on the GPU where gat_b200.run computed
    it and its statistics.  Result objects hold (matrix, column); the host copy is made once, when the first
    result is asked for its samples (output_counts_pattern, getSample, user code) -- outputResults never is."""

    def __init__(self, tensor, as_uint32, first_column=0):
        self._tensor = tensor
        self._as_uint32 = as_uint32
        self._host = None
        self.nsamples = int(tensor.shape[0])
        # a column-sharded run (gat_b200.run, exchange="columns") holds the columns
        # [first_column, first_column + ncolumns) of the annotation tracks on this rank
        self.first_column = int(first_column)
        self.ncolumns = int(tensor.shape[1])

    def host(self):
        if self._host is None:
            h = self._tensor.cpu().numpy()
            self._host = h.view(np.uint32) if self._as_uint32 else h
            self._tensor = None
        return self._host

    def column(self, index):
        local = index - self.first_column
        if not 0 <= local < self.ncolumns:
            raise RuntimeError("column-sharded run: the samples of annotation column %i live on another rank "
                               "(this rank holds columns %i..%i); run with exchange='allgather' to keep the whole "
                               "matrix on every rank" % (index, self.first_column, self.first_column + self.ncolumns - 1))
        return self.host()[:, local]

    def text(self):
        """-> (text uint8[], col_off): every column as b"c0,c1,..." (the counts-table format), formatted on
        the GPU (gatb_format_counts); integer counters only"""
        if not self._as_uint32:
            raise TypeError("float sample matrices are formatted on the host")
        if self._tensor is not None:
            return getContext().format_counts(device_ptr=self._tensor.data_ptr(), n_samples=self.nsamples,
                                              n_cols=int(self._tensor.shape[1]))
        return getContext().format_counts(counts=self._host)


class SamplesNotKept(SampleMatrix):
    """Stands in for the sample matrix of a run with keep_samples=False (gat_b200.run): the statistics were
    computed from slabs of samples that no longer exist, so the samples themselves cannot be handed out."""

    def __init__(self, nsamples, ncolumns):
        self._tensor = self._host = None
        self._as_uint32 = True
        self.nsamples = int(nsamples)
        self.first_column = 0
        self.ncolumns = int(ncolumns)

    def _refuse(self, *args):
        raise RuntimeError("the samples of this result were not kept (gat_b200.run with keep_samples=False computes "
                           "the statistics without the sample matrix); run with keep_samples=True to keep them")

    host = column = text = _refuse


class AnnotatorResult(object):
    """observed vs simulated counts of one (track, annotation, counter) with expected, CI95, stddev,
    fold, empirical p-value and q-value (gat/Engine.pyx:1725-1852).  The statistics are computed on
    the GPU (gatb_column_stats); `stats` lets gat_b200.run() pass in the row of a batched call."""

    format_expected = "%6.4f"
    format_fold = "%6.4f"
    format_pvalue = "%6.4e"
    format_counts = "%i"
    format_density = "%6.4e"

    headers = ["track", "annotation", "observed", "expected", "CI95low", "CI95high", "stddev", "fold",
               "l2fold", "pvalue", "qvalue"]

    def __init__(self, track, annotation, counter, observed, samples, reference=None, pseudo_count=1.0,
                 stats=None):
        self.track = track
        self.annotation = annotation
        self.counter = counter
        self.observed = float(observed)
        # the samples stay wherever they arrive -- a column of a SampleMatrix still on the GPU when built by
        # gat_b200.run, else an array -- and are converted to float64 only when asked for
        if isinstance(samples, tuple) and isinstance(samples[0], SampleMatrix):
            self._lazy, self._array = samples, None
            self.nsamples = samples[0].nsamples
        else:
            self._lazy = None
            self._array = samples if isinstance(samples, np.ndarray) else np.array(samples, dtype=np.float64)
            self.nsamples = len(self._array)
        self.format_observed = "%i"
        self.qvalue = 1.0
        if self.nsamples < 1:
            raise ValueError("no samples")
        if stats is None:
            col = self._column()
            ref = None if reference is None else [reference.fold]
            st = getContext().column_stats(col, [self.observed], pseudo_count=pseudo_count, ref_fold=ref)
            stats = dict((k, float(v[0])) for k, v in st.items())
        self.expected = stats["expected"]
        self.stddev = stats["stddev"]
        self.lower95 = stats["lower95"]
        self.upper95 = stats["upper95"]
        self.fold = stats["fold"]
        self.pvalue = stats["pvalue"]

    @property
    def _source(self):
        if self._array is None:
            self._array = self._lazy[0].column(self._lazy[1])
        return self._array

    def _column(self):
        """the samples as an (n,1) uint32 (integer counters) or float64 column for gatb_column_stats"""
        a = self._source
        if a.dtype.kind in "ui":
            return np.ascontiguousarray(a, dtype=np.uint32).reshape(-1, 1)
        a = np.asarray(a, dtype=np.float64)
        if np.all(a == np.floor(a)) and a.min() >= 0 and a.max() < 2 ** 32:
            return np.ascontiguousarray(a, dtype=np.uint32).reshape(-1, 1)
        return np.ascontiguousarray(a).reshape(-1, 1)

    @property
    def samples(self):
        return np.array(self._source, dtype=np.float64)

    def getSample(self, sample_id):
        return float(self._source[sample_id])

    def getEmpiricalPValue(self, value):
        # against the STORED expected value (gat/Engine.pyx:1564), which includes a reference fold
        return float(getContext().column_pvalue(self._column(), [float(value)], [self.expected])[0])

    def _columns(self):
        if self.fold > 0:
            logfold = self.format_fold % math.log(self.fold, 2)
        else:
            logfold = "-inf"
        return [self.track, self.annotation, self.format_observed % self.observed,
                self.format_expected % self.expected, self.format_expected % self.lower95,
                self.format_expected % self.upper95, self.format_expected % self.stddev,
                self.format_fold % self.fold, logfold, self.format_pvalue % self.pvalue,
                self.format_pvalue % self.qvalue]

    def __str__(self):
        return "\t".join(self._columns())


class AnnotatorResultExtended(AnnotatorResult):
    """AnnotatorResult plus size / overlap / density columns (gat/Engine.pyx:1854-1974)."""

    headers = AnnotatorResult.headers + [
        "track_nsegments", "track_size", "track_density",
        "annotation_nsegments", "annotation_size", "annotation_density",
        "overlap_nsegments", "overlap_size", "overlap_density",
        "percent_overlap_nsegments_track", "percent_overlap_size_track",
        "percent_overlap_nsegments_annotation", "percent_overlap_size_annotation"]

    def __init__(self, track, annotation, counter, observed, samples, track_segments, annotation_segments,
                 workspace, reference=None, pseudo_count=1.0, stats=None, sizes=None):
        """sizes: optional precomputed dict with track_nsegments, track_size, annotation_nsegments,
        annotation_size, overlap_nsegments, overlap_size, workspace_size (gat_b200.run computes them once per
        track / annotation, the overlap columns on the GPU via overlapColumns)"""
        AnnotatorResult.__init__(self, track, annotation, counter, observed, samples,
                                 reference=reference, pseudo_count=pseudo_count, stats=stats)
        if sizes is not None:
            for k in ("track_nsegments", "track_size", "annotation_nsegments", "annotation_size",
                      "overlap_nsegments", "overlap_size", "workspace_size"):
                setattr(self, k, sizes[k])
            return
        self.track_nsegments = track_segments.counts()
        self.track_size = track_segments.sum()
        self.annotation_nsegments = annotation_segments.counts()
        self.annotation_size = annotation_segments.sum()
        overlap = track_segments.clone()
        overlap.intersect(annotation_segments)
        self.overlap_nsegments = overlap.counts()
        self.overlap_size = overlap.sum()
        self.workspace_size = workspace.sum()

    def __str__(self):
        def pct(a, b, fmt):
            return fmt % (100.0 * float(a) / b) if b > 0 else "na"
        f, d, c = self.format_fold, self.format_density, self.format_counts
        return "\t".join(self._columns() + [
            c % self.track_nsegments, c % self.track_size, pct(self.track_size, self.workspace_size, d),
            c % self.annotation_nsegments, c % self.annotation_size,
            pct(self.annotation_size, self.workspace_size, d),
            c % self.overlap_nsegments, c % self.overlap_size, pct(self.overlap_size, self.workspace_size, d),
            pct(self.overlap_nsegments, self.track_nsegments, f), pct(self.overlap_size, self.track_size, f),
            pct(self.overlap_nsegments, self.annotation_nsegments, f),
            pct(self.overlap_size, self.annotation_size, f)])


# ------------------------------------------------------------------------------------ p / q values
def getNormedPValue(value, r):
    """p-value assuming normally distributed samples (gat/Engine.pyx:1976-1988)"""
    absval = abs(value - r.expected)
    if r.stddev == 0:
        return 1.0
    import scipy.stats
    return 1.0 - scipy.stats.norm.cdf(absval, 0, r.stddev)


def getEmpiricalPValue(value, r):
    return r.getEmpiricalPValue(value)


def updatePValues(annotator_results, method="empirical"):
    if method == "norm":
        f = getNormedPValue
    elif method == "empirical":
        f = getEmpiricalPValue
    else:
        raise ValueError("unknown method '%s'" % method)
    for r in annotator_results:
        r.pvalue = f(r.observed, r)


def getQValues(pvalues, method="storey", **kwargs):
    """q-values for a list of p-values (gat/Engine.pyx:2025-2039)"""
    if method == "storey":
        try:
            fdr = Stats.computeQValues(pvalues,
                                       vlambda=kwargs.get("vlambda", np.arange(0, 0.95, 0.05)),
                                       pi0_method=kwargs.get("pi0_method", "smoother"))
        except ValueError:
            return [1.0] * len(pvalues)
        return fdr.qvalues
    return Stats.adjustPValues(pvalues, method=method)


def updateQValues(annotator_results, method="storey", **kwargs):
    pvalues = [r.pvalue for r in annotator_results]
    for r, q in zip(annotator_results, getQValues(pvalues, method, **kwargs)):
        r.qvalue = q
