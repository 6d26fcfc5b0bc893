"""CPU: the host-side C++ of bin/match (readers, pruning, writer) against the oracle port and the
reference's documented quirks."""
import gzip
import os

import numpy as np
import pytest

from frog_b200 import hostio, pairsbin, synth
from oracle import oracle as O


def test_bin_reader_phantom_record(built, tmp_path):
    """match.cpp:184-205: `while(!feof)` appends one record whose six header fields all equal the
    last response and whose descriptor is zero."""
    kp = synth.make("iid", 37, 5)
    p = str(tmp_path / "a.bin")
    synth.write_bin(kp, p)
    head, desc = hostio.read_keypoints(p)
    assert head.shape == (38, 6) and desc.shape == (38, 48)
    assert np.array_equal(head[:37], kp.records()[:, :6]) and np.array_equal(desc[:37], kp.desc)
    assert np.all(head[37] == kp.response[-1]) and not desc[37].any()
    rec = O.PortLib().read_bin(p)
    assert np.array_equal(rec[:, :6], head) and np.array_equal(rec[:, 6:], desc)


def test_bin_reader_truncated_tail(built, tmp_path):
    kp = synth.make("iid", 5, 6)
    raw = kp.records().astype("<f4").tobytes()
    p = str(tmp_path / "t.bin")
    open(p, "wb").write(raw[:-100])  # cut inside the last descriptor
    head, desc = hostio.read_keypoints(p)
    rec = O.PortLib().read_bin(p)
    assert np.array_equal(rec[:, :6], head) and np.array_equal(rec[:, 6:], desc)
    assert head.shape[0] == 5  # the short read sets EOF: no phantom after a truncated record


def test_text_readers_match_port_and_bin(built, tmp_path):
    kp = synth.make("bank", 64, 2)
    pc, pg = str(tmp_path / "a.csv"), str(tmp_path / "a.csv.gz")
    synth.write_csv(kp, pc)
    synth.write_csv_gz(kp, pg)
    hc, dc = hostio.read_keypoints(pc)
    hg, dg = hostio.read_keypoints(pg)
    assert np.array_equal(hc, hg) and np.array_equal(dc, dg)
    assert np.array_equal(hc, kp.records()[:, :6]) and np.array_equal(dc, kp.desc)
    rec = O.PortLib().parse_csv(gzip.open(pg).read())
    assert np.array_equal(rec[:, :6], hc) and np.array_equal(rec[:, 6:], dc)


def test_csv_quirks(built, golden_dir):
    """CRLF, exponent cells, leading blanks, trailing commas, short and empty lines."""
    head, desc = hostio.read_keypoints(os.path.join(golden_dir, "quirks.csv"))
    rec = O.PortLib().parse_csv(open(os.path.join(golden_dir, "quirks.csv"), "rb").read())
    assert head.shape[0] == 40
    assert np.array_equal(rec[:, :6], head) and np.array_equal(rec[:, 6:], desc)


def test_prune_and_zfilter(built):
    kp = synth.make("iid", 500, 9)
    rec = kp.records()
    head, desc = hostio.filter_prune(rec[:, :6], rec[:, 6:], zT=10.0, zmin=200.0, zmax=900.0, sp=1000.0, np_keep=50)
    z = rec[:, 2] + np.float32(10.0)
    keep = ~((z < 200.0) | (z > 900.0)) & ~(rec[:, 5] < 1000.0)
    assert head.shape[0] == 50
    # survivors are the 50 largest responses of the kept set (order is libstdc++'s, pinned by golden bin_prune)
    assert set(head[:, 5].tolist()) == set(np.sort(rec[keep, 5])[::-1][:50].tolist())


def test_writer_layout(built, tmp_path):
    heads = [np.arange(12, dtype=np.float32).reshape(2, 6), np.zeros((0, 6), np.float32)]
    blocks = [(0, 1, np.array([[1, 0]], np.uint32)), (65536 + 3, 1, np.zeros((0, 2), np.uint32))]
    p = str(tmp_path / "w.bin")
    hostio.write_pairs_bin(p, ["/x/y/a.bin", "b\\c.csv"], [[1.0, 2.0, 3.0], [0, 0, 0]], heads, blocks)
    pf = pairsbin.parse(p)
    assert pf.names == ["a.bin", "c.csv"] and pf.rigids[0] == (1.0, 2.0, 3.0)
    assert [b[:2] for b in pf.blocks] == [(0, 1), (3, 1)]  # ids truncated to u16 (match.cpp:735-736)
    assert pf.blocks[1][2].shape == (0, 2)  # empty blocks are still written (match.cpp:732-738)


def test_fast_decimal_parser_is_strtof(built):
    """keypoint_io.cpp fast_strtof: the libc-free text->float path must agree with strtof (= std::stof,
    match.cpp:69,152) bit for bit, value and consumed prefix, on surf3d-style "%f" cells, long digit
    strings, exponent forms (also broken ones), exact float midpoints and odd shapes."""
    import ctypes as C

    from frog_b200 import build
    L = C.CDLL(build.FMIO)
    L.fmio_fuzz_floats.argtypes = [C.c_uint64, C.c_int64, C.POINTER(C.c_int64), C.c_char_p, C.c_size_t]
    L.fmio_fuzz_floats.restype = C.c_int64
    n_fast, bad = C.c_int64(), C.create_string_buffer(128)
    for seed in (1, 2, 3):
        n_bad = L.fmio_fuzz_floats(seed, 400_000, C.byref(n_fast), bad, 128)
        assert n_bad == 0, f"first mismatching cell: {bad.value!r}"
        assert n_fast.value > 200_000  # the fast path really carries the common formats


def test_csv_long_descriptors_through_cli_readers(tmp_path):
    """surf3d -type 2 writes 8 r^3 = 1000 values per keypoint at the default radius (vtkOpenSURF3D/surf3d.cxx:36-39);
    the CSV readers take whatever length the rows have (match.cpp:160-168)."""
    import gzip
    rng = np.random.default_rng(3)
    n, d = 17, 1000
    rec = np.concatenate([rng.uniform(0, 100, (n, 6)), rng.standard_normal((n, d))], axis=1).astype(np.float32)
    text = "\n".join(",".join("%f" % v for v in row) for row in rec) + "\n"
    p_csv, p_gz = tmp_path / "long.csv", tmp_path / "long.csv.gz"
    p_csv.write_text(text)
    with gzip.open(p_gz, "wt") as f:
        f.write(text)
    want = np.array([[np.float32(float("%f" % v)) for v in row] for row in rec], np.float32)
    for p in (p_csv, p_gz):
        head, desc = hostio.read_keypoints(str(p))
        assert head.shape == (n, 6) and desc.shape == (n, d)
        assert np.array_equal(head, want[:, :6]) and np.array_equal(desc, want[:, 6:])


def _fast_inflate(raw: bytes, cap: int):
    import ctypes as C
    from frog_b200 import build
    L = C.CDLL(build.FMIO)
    L.fmio_fast_inflate.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
    out = C.create_string_buffer(cap + 1)
    got = C.c_size_t(0)
    rc = L.fmio_fast_inflate(raw, len(raw), out, cap, C.byref(got))
    return rc, out.raw[:got.value]


def test_fast_inflate_equals_zlib(built):
    """fast_inflate.cpp (the decoder behind the .csv.gz reader) against zlib: every block type (stored, fixed, dynamic),
    every compression level and strategy, code lengths up to 15 bits, sync/full flush points, a gzip header with a
    file name, sizes around the 258-byte match and 64 KiB stored-block limits."""
    import gzip
    import io
    import zlib
    rng = np.random.default_rng(2)
    probs = np.array([2.0 ** -i for i in range(1, 40)])
    probs /= probs.sum()
    fib = [1, 1]
    while len(fib) < 30:
        fib.append(fib[-1] + fib[-2])
    corpus = [b"", b"a", b"hello, hello, hello, hello\n" * 3, bytes(range(256)) * 5,
              rng.integers(0, 256, 100000, dtype=np.uint8).tobytes(), rng.integers(0, 4, 300000, dtype=np.uint8).tobytes(),
              b"\0" * 1000000, ("%f,%f,%d\n" % (1.5, -2.25, 7)).encode() * 50000,
              ",".join("%f" % v for v in rng.standard_normal(100000)).encode(),
              bytes(rng.choice(39, 400000, p=probs).astype(np.uint8) + 40),
              b"".join(bytes([65 + i]) * f for i, f in enumerate(fib))]
    corpus += [bytes(rng.integers(97, 101, n, dtype=np.uint8)) for n in (1, 2, 3, 7, 8, 9, 257, 258, 259, 65535, 65536, 65537)]
    n_ok = 0
    for data in corpus:
        for level in (0, 1, 6, 9):
            for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE):
                co = zlib.compressobj(level, zlib.DEFLATED, 31, 9, strategy)
                raw = co.compress(data) + co.flush()
                rc, got = _fast_inflate(raw, len(data) + 16)
                assert rc == 1 and got == data, (len(data), level, strategy)
                n_ok += 1
        bio = io.BytesIO()
        with gzip.GzipFile(filename="points.csv", mode="wb", fileobj=bio, compresslevel=6) as f:
            f.write(data)
        rc, got = _fast_inflate(bio.getvalue(), len(data) + 16)
        assert rc == 1 and got == data
        co = zlib.compressobj(6, zlib.DEFLATED, 31)
        step = max(1, len(data) // 7)
        raw = b"".join(co.compress(data[i:i + step]) + co.flush(zlib.Z_SYNC_FLUSH if (i // step) % 2 else zlib.Z_FULL_FLUSH)
                       for i in range(0, len(data), step)) + co.flush()
        rc, got = _fast_inflate(raw, len(data) + 16)
        assert rc == 1 and got == data
    assert n_ok == len(corpus) * 16


def test_fast_inflate_declines_what_it_cannot_vouch_for(built, tmp_path):
    """Truncated, corrupted, multi-member or trailing-garbage input: the fast decoder says no (or, for a flipped bit
    zlib does not mind either, yields zlib's bytes) and the reader falls back to zlib -- same keypoints as before."""
    import random
    import zlib
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    text = b"".join(b"%d.5,2,3,1.5,0,9,0.25,0.5\n" % i for i in range(3000))
    good = co.compress(text) + co.flush()
    bad = [good[:-1], good[:len(good) // 2], good + good, good + b"x", good[:-8] + b"\0\0\0\0" + good[-4:],
           good[:-4] + b"\1\0\0\0", b"\x1f\x8b\x08", b"", b"not gzip at all" * 10]
    r = random.Random(1)
    for _ in range(60):
        b = bytearray(good)
        b[r.randrange(10, len(good) - 8)] ^= 1 << r.randrange(8)
        bad.append(bytes(b))
    declined = 0
    for b in bad:
        rc, got = _fast_inflate(b, 400000)
        if rc == 1:
            assert zlib.decompress(b, 47) == got
        else:
            declined += 1
    assert declined >= len(bad) - 3
    # Two members: like boost's gzip_decompressor (match.cpp:55-58) the reader continues into the second one.
    # Trailing garbage / a truncated member: everything that could be inflated, minus an unterminated last line.
    for name, payload, rows in (("two.csv.gz", good + good, 6000), ("junk.csv.gz", good + b"garbage", 3000)):
        p = tmp_path / name
        p.write_bytes(payload)
        head, desc = hostio.read_keypoints(str(p))
        assert head.shape == (rows, 6) and desc.shape == (rows, 2) and head[7, 0] == 7.5
        assert head[rows - 1, 0] == 2999.5
    p = tmp_path / "cut.csv.gz"
    p.write_bytes(good[:len(good) // 2])
    head, desc = hostio.read_keypoints(str(p))
    n = head.shape[0]
    assert 0 < n < 3000 and np.array_equal(head[:, 0], np.arange(n) + 0.5) and desc.shape == (n, 2)


def test_multi_member_gzip_matches_the_reference_build(built, tmp_path):
    """A .csv.gz made of two concatenated members loads as the concatenation of both texts -- in this reader and in the
    verbatim reference build (whose Boost stand-in, oracle/shim, continues into following members as Boost does) --
    run where oracle/_ref is built, else as recorded in tests/golden/ref."""
    import sys
    from frog_b200 import pairsbin
    from oracle import oracle as O
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_ref_golden as rg
    two, lst, b = rg.multi_member_files(str(tmp_path))
    head, desc = hostio.read_keypoints(two)
    assert desc.shape == (65, 48) and np.array_equal(desc[40:], b.desc)
    if os.path.exists(O.REF_BIN):
        O.run_ref_binary([lst, "-o", str(tmp_path / "ref.bin"), "-d", "1"])
        ref_points = pairsbin.parse(str(tmp_path / "ref.bin")).points[0]
    else:
        ref_points = rg.load("multi_member")[1]["points0"]
    assert ref_points.shape[0] == 65 and np.array_equal(ref_points, head)


def test_text_writer_matches_printf(built, tmp_path):
    """The bench's C text writer (fmio_write_csv) prints "%f" exactly as printf does; the files it writes hold the same
    text as the Python writer's."""
    import gzip
    from frog_b200 import synth
    assert hostio.load().fmio_fuzz_fmt(3, 2_000_000) == 0
    kp = synth.make("iid", 300, 5)
    synth.write_csv_gz(kp, str(tmp_path / "a.csv.gz"))
    synth._write_fast(kp, str(tmp_path / "b.csv.gz"), "csv.gz")
    assert gzip.open(tmp_path / "a.csv.gz").read() == gzip.open(tmp_path / "b.csv.gz").read()
    synth.write_csv(kp, str(tmp_path / "a.csv"))
    synth._write_fast(kp, str(tmp_path / "b.csv"), "csv")
    assert (tmp_path / "a.csv").read_bytes() == (tmp_path / "b.csv").read_bytes()


def test_descriptor_cells_are_strtof_on_every_value(built, tmp_path):
    """The eight-bytes-at-a-time path for "%f" descriptor cells (`-?0.dddddd`): ALL 10^6 values, both signs, parsed
    through the row loop and compared bit for bit with libc's strtof; and cells that only look like descriptor cells
    fall through to the general path with the same result as before."""
    import ctypes as C
    libc = C.CDLL("libc.so.6")
    libc.strtof.restype = C.c_float
    libc.strtof.argtypes = [C.c_char_p, C.c_void_p]
    vals = np.arange(1000000)
    cells = np.char.add("0.", np.char.zfill(vals.astype(str), 6))
    rng = np.random.default_rng(11)
    neg = rng.random(1000000) < 0.5
    cells = np.where(neg, np.char.add("-", cells), cells)
    rows = cells.reshape(-1, 50)  # 6 header cells + 44 descriptor cells per row
    text = "\n".join(",".join(r) for r in rows) + "\n"
    path = str(tmp_path / "all.csv")
    open(path, "w").write(text)
    head, desc = hostio.read_keypoints(path, d_cap=64)
    got = np.concatenate([head, desc], 1).reshape(-1)
    assert got.size == 1000000
    want = np.array([libc.strtof(c.encode(), None) for c in cells.tolist()], np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.signbit(got[vals == 0][neg[vals == 0]]).all()  # "-0.000000" keeps its sign
    # near misses of the shape: seven decimals, exponent, a space, a hex digit, "1." instead of "0.", a short last cell
    odd = ["0.1234567", "0.12345e1", "0.12 456", "0.12a456", "1.234567", "-1.000000", "0.123456 ", "+0.123456", "0.5"]
    line = ",".join(["1", "2", "3", "4", "5", "6"] + odd) + "\n"
    open(path, "w").write(line * 3)
    head, desc = hostio.read_keypoints(path, d_cap=64)
    want = np.array([libc.strtof(c.encode(), None) for c in odd], np.float32)
    assert desc.shape == (3, len(odd)) and np.array_equal(desc[1].view(np.uint32), want.view(np.uint32))
