"""The GPU reader of counts tables (gatb_parse_counts, Engine.readCountsTable) and gat-compare on device matrices
(gatb_compare_stats_device): the same results as the host reader, or the same exception, on every input.

The bodies that take only `ctx` also run on the emulated kernels (tests/test_emu_counts_table.py); there "device"
memory is host memory, which _Dev hides."""
import gzip
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HEADER = b"track\tannotation\tobserved\tcounts\n"
STATS = ["expected", "stddev", "lower95", "upper95", "fold", "pvalue"]


def _emulated(ctx):
    return hasattr(ctx.lib, "gatb_emulation_marker")


class _Dev(object):
    """a copy of a host array in the context's device memory (a host copy for the emulated kernels)"""

    def __init__(self, ctx, array):
        array = np.ascontiguousarray(array)
        if _emulated(ctx):
            self.obj = array.copy() if array.size else np.zeros(1, dtype=array.dtype)
            self.ptr = self.obj.ctypes.data
        else:
            import torch
            self.obj = torch.from_numpy(array.copy() if array.size else np.zeros(1, dtype=array.dtype)).to("cuda")
            self.ptr = self.obj.data_ptr()

    def host(self):
        return self.obj if isinstance(self.obj, np.ndarray) else self.obj.cpu().numpy()


def parse(ctx, body):
    """-> (table dict of Context.parse_counts, uint32 matrix [n_samples][n_rows] or None)"""
    text = _Dev(ctx, np.frombuffer(body, dtype=np.uint8))
    table = ctx.parse_counts(text.ptr, len(body), body.count(b"\n"))
    if not table["plain"] or table["n_rows"] == 0:
        return table, None
    out = _Dev(ctx, np.zeros((table["n_samples"], table["n_rows"]), dtype=np.uint32))
    ctx.parse_counts(text.ptr, len(body), body.count(b"\n"), counts_ptr=out.ptr)
    return table, out.host().view(np.uint32)


_LINE = re.compile(rb"[^\t\n\r]*\t[^\t\n\r]*\t[^\t\n\r]*\t([0-9]{1,10}(?:,[0-9]{1,10})*)\n")


def reference(body):
    """the grammar of gatb_parse_counts restated in Python -> (line table, matrix) or None when not plain"""
    if not body or b"\r" in body or not body.endswith(b"\n"):
        return None
    lines, cols, pos = [], [], 0
    for line in body.split(b"\n")[:-1]:
        m = _LINE.fullmatch(line + b"\n")
        if not m:
            return None
        vals = [int(x) for x in m.group(1).split(b",")]
        if max(vals) >= 2 ** 32:
            return None
        lines.append((pos, pos + m.start(1)))
        cols.append(vals)
        pos += len(line) + 1
    if len(set(len(c) for c in cols)) != 1:
        return None
    return np.array(lines, dtype=np.uint64), np.array(cols, dtype=np.uint32).T.copy()


def first_offending(body):
    r"""the offset gatb_parse_counts reports for a body that is not plain (None: plain): the first '\r', the start of a
    last line without '\n', a line's '\n' before its third tab, its fourth tab, in a counts field a byte other than a
    digit or a ',' / '\n' after a digit, the start of a number of more than 10 digits or >= 2^32, a comma that starts
    a value past the first line's number of values, and the '\n' of a line with fewer values than the first line"""
    if not body:
        return None
    found = []
    if b"\r" in body:
        found.append(body.index(b"\r"))
    last = body.rfind(b"\n")
    if last != len(body) - 1:
        found.append(last + 1)
    pos, n_values = 0, None
    for k, line in enumerate(body[:last + 1].split(b"\n")[:-1]):
        tabs = [i for i, c in enumerate(line) if c == 9]
        end = pos + len(line)
        if len(tabs) < 3:
            found.append(end)
        else:
            if len(tabs) > 3:
                found.append(pos + tabs[3])
            cs = tabs[2] + 1
            field = line[cs:] + b"\n"
            if k == 0:
                n_values = field.count(b",") + 1
            commas = 0
            for j, c in enumerate(field):
                prev_digit = j > 0 and field[j - 1:j].isdigit()
                if field[j:j + 1].isdigit():
                    if not prev_digit:
                        d = 0
                        while d < 11 and field[j + d:j + d + 1].isdigit():
                            d += 1
                        if d > 10 or int(field[j:j + d]) >= 2 ** 32:
                            found.append(pos + cs + j)
                elif c not in b",\n" or not prev_digit or (c == 44 and n_values and commas == n_values - 1):
                    found.append(pos + cs + j)
                commas += c == 44
            if len(tabs) == 3 and n_values and field.count(b",") < n_values - 1:
                found.append(end)
        pos = end + 1
    return min(found) if found else None


def check_against_reference(ctx, body):
    table, matrix = parse(ctx, body)
    ref = reference(body)
    bad = first_offending(body)
    assert (bad is None) == (ref is not None), body[:200]
    assert table["plain"] == (ref is not None), body[:200]
    if ref is None:
        assert table["bad_offset"] == bad, body[:200]
        return table
    assert table["bad_offset"] == 2 ** 64 - 1
    assert table["n_rows"] == ref[1].shape[1] and table["n_samples"] == ref[1].shape[0]
    assert np.array_equal(table["lines"], ref[0])
    assert matrix.dtype == np.uint32 and np.array_equal(matrix, ref[1])
    return table


# ----------------------------------------------------------------------------------- bodies (GPU and emulated)
EDGE_BODIES = [
    b"t\ta\t1\t7\n",                                              # 1 sample, 1 row
    b"t\ta\t3\t0,4294967295,0000000007\nu\tb\t2\t1,2,3\n",      # the extreme values, leading zeros
    b"t\ta\t1\t4294967296\n",                                     # >= 2^32
    b"t\ta\t1\t1.5\n",                                            # a float
    b"t\ta\t1\t1,2\r\nt\tb\t1\t3,4\r\n",                         # \r\n
    b"t\ta\t1\t1,2\nt\tb\t1\t3,4",                                # no final newline
    b"t\ta\t1\t1,2\n\nt\tb\t1\t3,4\n",                           # an empty line
    b"t\ta\t1\t1,2\t5\n",                                         # a fourth tab
    b"t\ta\t1\t1,,2\n",                                           # ,,
    b"t\ta\t1\t1,2,\n",                                           # a trailing comma
    b"t\ta\t1\t,1,2\n",                                           # a leading comma
    b"t\ta\t1\t\n",                                               # an empty counts field
    b"t\ta\t1\n",                                                 # two tabs
    b"t\ta\t1\t1,2\nt\tb\t1\t1,2,3\n",                           # ragged rows
    b"t\ta\t1\t1,2,3\nt\tb\t1\t1,2\nt\tc\t1\t1,2,3,4\n",           # ragged rows, fewer then more
    b"t\ta\t1\t1,2\nt\tb\t1\t1,2,3\t4\n",                       # more values and a fourth tab
    b"t\ta\t1\t00000000007\n",                                    # 11 digits
    b"t\ta\t1\t+1\n",
    b"t\ta\t1\t1 \n",
    "träck\tanno,ü中\t1e3\t5,6\n".encode("utf-8"),  # non-ASCII names, a comma in a name
]


def test_parse_grammar_edges(ctx):
    for body in EDGE_BODIES:
        check_against_reference(ctx, body)
    # the offending byte of a few bodies
    assert parse(ctx, b"t\ta\t1\t1,,2\n")[0]["bad_offset"] == 8
    assert parse(ctx, b"t\ta\t1\t1,2\t5\n")[0]["bad_offset"] == 9
    assert parse(ctx, b"t\ta\t1\t1\r\n")[0]["bad_offset"] == 7
    assert parse(ctx, b"t\ta\t1\t1,2\nt\tb\t1\t1\n")[0]["bad_offset"] == 17       # fewer values: the '\n'
    assert parse(ctx, b"t\ta\t1\t1\nt\tb\t1\t1,2,3\n")[0]["bad_offset"] == 15      # more: the first extra ','
    assert parse(ctx, b"t\ta\t1\t1\nt\tb")[0]["bad_offset"] == 8
    empty = parse(ctx, b"")[0]
    assert empty["plain"] and empty["n_rows"] == 0


def test_parse_tile_edges(ctx):
    """every byte of a line -- digits, commas, tabs, the newline -- on either side of a tile edge"""
    tile = 4096                                                   # PARSE_TILE (count.cu)
    rest = b"\tann\t12\t4294967295,0,17,123456789,0000000001\n"
    filler = b"f\tg\t1\t" + b",".join([b"99999"] * 5) + b"\n"
    for edge in (tile, 2 * tile):
        head = filler * ((edge - 64) // len(filler))
        for s in range(len(rest) + 1):
            # the line's track name pads it so that byte s of `rest` is the first byte of the next tile
            body = head + b"x" * (edge - len(head) - s) + rest + filler
            assert body[edge:edge + 1] == (rest + filler)[s:s + 1]
            check_against_reference(ctx, body)
    # a number running over the edge by up to 10 digits, and an 11th digit just past it
    for d in range(1, 12):
        body = b"x" * (tile - 5 - d // 2) + b"\ta\t1\t" + b"7" * d + b"\n"
        check_against_reference(ctx, body)


def test_parse_random_tables(ctx):
    rng = np.random.default_rng(11)
    size = 60000 if _emulated(ctx) else 4 << 20
    for trial in range(3):
        n_samples = int(rng.integers(1, 400))
        vals = []
        body = b""
        while len(body) < size:
            v = rng.integers(0, 2 ** 32, size=n_samples, dtype=np.uint64) >> rng.integers(0, 33, size=n_samples).astype(np.uint64)
            name = b"n" * int(rng.integers(0, 50))
            body += b"%s\tanno%d\t%d\t%s\n" % (name, len(vals), int(v[0]), b",".join(b"%d" % x for x in v.tolist()))
            vals.append(v)
        check_against_reference(ctx, body)
        # one random byte damaged: same verdict and offending byte as the reference
        for i in rng.integers(0, len(body), size=4).tolist():
            for c in (b",", b"\t", b"\n", b"a", b"\r", b"5"):
                check_against_reference(ctx, body[:i] + c + body[i + 1:])


def test_compare_stats_device_equals_host(ctx):
    """gatb_compare_stats_device on uint32 (and mixed uint32 / float64) device matrices == gatb_compare_stats on the
    same values as float64 host matrices, all six outputs, bit for bit"""
    rng = np.random.default_rng(5)
    S = 300 if _emulated(ctx) else 20000
    m1 = rng.poisson(50, size=(S, 6)).astype(np.uint32)
    m2 = rng.poisson(40, size=(S, 4)).astype(np.uint32)
    m2[:, 0] = 0
    c1, c2 = np.array([0, 1, 2, 5, 3], dtype=np.int32), np.array([0, 1, 3, 2, 0], dtype=np.int32)
    obs1, obs2 = rng.uniform(10, 90, 5), rng.uniform(10, 90, 5)
    delta = rng.normal(size=5)
    host = ctx.compare_stats(m1.astype(np.float64), m2.astype(np.float64), c1, c2, obs1, obs2, delta, pseudo_count=1.0)
    d1, d2 = _Dev(ctx, m1), _Dev(ctx, m2)
    f2 = _Dev(ctx, m2.astype(np.float64))
    for a, b in (((d1.ptr, S, 6, 0), (d2.ptr, S, 4, 0)), ((d1.ptr, S, 6, 0), (f2.ptr, S, 4, 1))):
        got = ctx.compare_stats(a, b, c1, c2, obs1, obs2, delta, pseudo_count=1.0)
        for k in STATS:
            assert np.array_equal(got[k], host[k], equal_nan=True), k
    # one matrix against itself
    host1 = ctx.compare_stats(m1.astype(np.float64), None, c1, c1, obs1, obs2, delta)
    got1 = ctx.compare_stats((d1.ptr, S, 6, 0), None, c1, c1, obs1, obs2, delta)
    for k in STATS:
        assert np.array_equal(got1[k], host1[k], equal_nan=True), k


# ----------------------------------------------------------------------------------- the readers (GPU only)
def _results(rs):
    return [(r.track, r.annotation, r.observed, r.nsamples, list(r.samples)) + tuple(getattr(r, k) for k in
            ("expected", "stddev", "lower95", "upper95", "fold", "pvalue")) for r in rs]


def _outcome(fn, *args):
    try:
        return "ok", fn(*args)
    except Exception as e:                                      # noqa: BLE001  (the exception is the result)
        return type(e), str(e)


def _write(path, data):
    if str(path).endswith(".gz"):
        with gzip.open(str(path), "wb") as f:
            f.write(data)
    else:
        with open(str(path), "wb") as f:
            f.write(data)
    return str(path)


def _readers_agree(path):
    import gat_b200
    from gat_b200 import compare
    a, b = _outcome(gat_b200.fromCounts, path), _outcome(gat_b200._fromCountsHost, path)
    assert a[0] == b[0] and (a[1] == b[1] if a[0] != "ok" else _results(a[1]) == _results(b[1])), path
    a, b = _outcome(compare.fromCountsBatched, path), _outcome(compare._fromCountsHost, path)
    assert a[0] == b[0], path
    if a[0] != "ok":
        assert a[1] == b[1]
    else:
        assert _results(a[1][0]) == _results(b[1][0])
        ma, mb = a[1][1], b[1][1]
        assert np.array_equal(ma.host() if hasattr(ma, "host") else ma, mb)


def test_readers_agree_on_grammar_edges(ctx, tmp_path):
    bodies = EDGE_BODIES + [b""]
    for i, body in enumerate(bodies):
        for suffix in (".tsv", ".tsv.gz"):
            _readers_agree(_write(tmp_path / ("t%d%s" % (i, suffix)), HEADER + body))
    _readers_agree(_write(tmp_path / "crlf.tsv", HEADER.replace(b"\n", b"\r\n") + b"t\ta\t1\t1,2\r\n"))
    _readers_agree(_write(tmp_path / "bad.tsv", b"track\tannotation\tobserved\n" + b"t\ta\t1\t1,2\n"))
    _readers_agree(_write(tmp_path / "obs.tsv", HEADER + b"t\ta\tx\t1,2\n"))
    from gat_b200 import engine as Engine
    assert Engine.readCountsTable(_write(tmp_path / "plain.tsv", HEADER + EDGE_BODIES[1])) is not None
    assert Engine.readCountsTable(_write(tmp_path / "float.tsv", HEADER + EDGE_BODIES[3])) is None


def test_counts_table_round_trip(ctx, tmp_path):
    """run() writes the tables of the integer counters; the GPU reader gives back the run's matrix exactly, and
    fromCounts the host reader's statistics"""
    import gat_b200
    from gat_b200 import engine as Engine, synthetic
    segments, annotations, workspaces, _ = synthetic.make(n_segments=300, n_annotations=5, n_annotation_intervals=400)
    workspace = synthetic.prepare(segments, annotations, workspaces)
    counters = [Engine.CounterNucleotideOverlap(), Engine.CounterSegmentOverlap()]
    for suffix in (".tsv", ".tsv.gz"):
        Engine.seed(3)
        pattern = str(tmp_path / ("counts_%s" + suffix))
        res = gat_b200.run(segments, annotations, workspace, Engine.SamplerAnnotator(), counters,
                           Engine.UnconditionalWorkspace(), num_samples=500, output_counts_pattern=pattern)
        for counter in ("nucleotide-overlap", "segment-overlap"):
            mine = [r for r in res if r.counter == counter]
            rows, matrix = Engine.readCountsTable(pattern % counter)
            assert [(t, a) for t, a, _ in rows] == [(r.track, r.annotation) for r in mine]
            assert np.array_equal(matrix.host(), np.stack([r.samples for r in mine], axis=1).astype(np.uint32))
            back, host = gat_b200.fromCounts(pattern % counter), gat_b200._fromCountsHost(pattern % counter)
            assert _results(back) == _results(host)
            for a, b in zip(back, host):
                assert a.getSample(7) == b.getSample(7) and a.getEmpiricalPValue(a.observed) == b.getEmpiricalPValue(b.observed)


def _table(rng, names, n_samples):
    return HEADER + b"".join(b"merged\t%s\t%d\t%s\n" % (n.encode(), int(rng.integers(5, 60)),
                                                        b",".join(b"%d" % v for v in rng.poisson(30, n_samples)))
                             for n in names)


def test_cli_output_same_with_either_reader(ctx, tmp_path, monkeypatch):
    """python -m gat_b200.compare (one and two files) and gat_b200.cli --input-counts-file print byte-identical
    tables with the GPU reader and with the host reader; ragged rows still raise in gat-compare"""
    from gat_b200 import cli, compare, engine as Engine
    rng = np.random.default_rng(2)
    f1 = _write(tmp_path / "c1.tsv", _table(rng, ["a%d" % i for i in range(6)], 700))
    f2 = _write(tmp_path / "c2.tsv.gz", _table(rng, ["a%d" % i for i in range(2, 9)], 700))
    reader = Engine.readCountsTable

    def outputs():
        out = []
        for k, args in enumerate([[f1], [f1, f2], ["--pvalue-method=norm", f2, f1]]):
            path = str(tmp_path / ("cmp%d.tsv" % k))
            assert compare.main(["gat-compare"] + args + ["--stdout=" + path]) == 0
            out.append(open(path, "rb").read())
        path = str(tmp_path / "cli.tsv")
        assert cli.main(["gat-run", "--input-counts-file=" + f1, "--stdout=" + path, "-v", "0"]) == 0
        out.append(open(path, "rb").read())
        return out

    seen = []
    monkeypatch.setattr(Engine, "readCountsTable", lambda fn: seen.append(fn) or reader(fn))
    device = outputs()
    assert seen and all(reader(fn) is not None for fn in (f1, f2))
    monkeypatch.setattr(Engine, "readCountsTable", lambda fn: None)
    host = outputs()
    assert device == host and all(len(x.splitlines()) > 1 for x in device)
    monkeypatch.setattr(Engine, "readCountsTable", reader)
    ragged = _write(tmp_path / "ragged.tsv", HEADER + b"t\ta\t1\t1,2\nt\tb\t1\t1,2,3\n")
    with pytest.raises(ValueError, match="rows differ in the number of samples"):
        compare.main(["gat-compare", ragged, "--stdout=" + str(tmp_path / "r.tsv")])


def test_compare_pairs_of_a_device_and_a_host_matrix(ctx, tmp_path, monkeypatch):
    """gat-compare on a table the GPU reader takes and one it leaves to the host reader (float values, '\r\n'): the
    same printed table as with the host reader for both; and Context.compare_stats on such mixed pairs"""
    import torch
    from gat_b200 import compare, engine as Engine
    rng = np.random.default_rng(9)
    names = ["a%d" % i for i in range(5)]
    plain = _write(tmp_path / "plain.tsv", _table(rng, names, 300))
    floats = _table(rng, names, 300).replace(b"\n", b".5\n").replace(b"counts.5\n", b"counts\n")
    f_float = _write(tmp_path / "float.tsv.gz", floats)
    f_crlf = _write(tmp_path / "crlf.tsv", _table(rng, names, 300).replace(b"\n", b"\r\n"))
    assert Engine.readCountsTable(plain) is not None
    assert Engine.readCountsTable(f_float) is None and Engine.readCountsTable(f_crlf) is None
    reader = Engine.readCountsTable
    cases = [[plain, f_float], [f_float, plain], [plain, f_crlf], [f_crlf, plain, f_float]]

    def outputs():
        out = []
        for k, files in enumerate(cases):
            path = str(tmp_path / ("mixed%d.tsv" % k))
            assert compare.main(["gat-compare"] + files + ["--stdout=" + path]) == 0
            out.append(open(path, "rb").read())
        return out

    device = outputs()
    monkeypatch.setattr(Engine, "readCountsTable", lambda fn: None)
    host = outputs()
    monkeypatch.setattr(Engine, "readCountsTable", reader)
    assert device == host and all(len(x.splitlines()) > 1 for x in device)
    # a device matrix against a host array, and against a SampleMatrix whose samples were copied to the host
    m1 = rng.poisson(30, size=(400, 4)).astype(np.uint32)
    m2 = rng.poisson(30, size=(400, 3)).astype(np.float64) + 0.25
    c1, c2 = np.array([0, 3, 1], dtype=np.int32), np.array([2, 0, 1], dtype=np.int32)
    args = (c1, c2, rng.uniform(10, 50, 3), rng.uniform(10, 50, 3), rng.normal(size=3))
    want = ctx.compare_stats(m1.astype(np.float64), m2, *args)
    d1 = _Dev(ctx, m1)
    moved = Engine.SampleMatrix(torch.from_numpy(m1.view(np.int32)).to("cuda"), True)
    moved.host()
    for a, b in (((d1.ptr, 400, 4, 0), m2), (moved, _Dev(ctx, m2))):
        b = (b.ptr, 400, 3, 1) if isinstance(b, _Dev) else b
        got = ctx.compare_stats(a, b, *args)
        for k in STATS:
            assert np.array_equal(got[k], want[k], equal_nan=True), k
