"""CPU: bin/surf3d's MetaImage reader (libfsio's fsio_read_metaimage) on every element type and every encoding it
accepts -- compressed (zlib or gzip wrapper, with and without CompressedDataSize), detached data files with
HeaderSize, big-endian data -- and its refusals."""
import os
import subprocess
import zlib

import numpy as np
import pytest

from frog_b200 import build, surf

SPACING, ORIGIN = (0.5, 0.75, 2.0), (1.0, -2.0, 3.5)


def source(dtype, shape=(5, 6, 7), seed=0):
    """Values that use each type's range: negative int8, uint32 above INT_MAX, doubles that are not floats."""
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    if dt.kind in "iu":
        info = np.iinfo(dt)
        return rng.integers(info.min, info.max, shape, dtype=dt, endpoint=True)
    return (rng.standard_normal(shape) * 1000).astype(dt)


ENCODINGS = {
    "local_raw": dict(),
    "local_zlib1": dict(compress=1),
    "local_zlib6": dict(compress=6),
    "local_zlib9": dict(compress=9),
    "local_gzip": dict(compress=6, gzip=True),
    "local_zlib_nosize": dict(compress=6, compressed_size=False),
    "local_gzip_nosize": dict(compress=6, gzip=True, compressed_size=False),
    "raw_header0": dict(data_file="d.raw", header_size=0),
    "raw_header37": dict(data_file="d.raw", header_size=37),
    "raw_header_auto": dict(data_file="d.raw", header_size=-1),
    "raw_no_headersize": dict(data_file="d.raw"),
    "zraw": dict(data_file="d.zraw", compress=6),
    "zraw_nosize_header13": dict(data_file="d.zraw", compress=1, compressed_size=False, header_size=13),
    "big_endian": dict(byte_order=">"),
    "big_endian_zlib": dict(byte_order=">", compress=6),
    "big_endian_zraw": dict(byte_order=">", compress=9, data_file="d.zraw"),
}
DTYPES = [np.uint8, np.int8, np.int16, np.uint16, np.int32, np.uint32, np.float32, np.float64]


@pytest.mark.parametrize("enc", sorted(ENCODINGS))
@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: np.dtype(d).name)
def test_every_type_and_encoding(built, tmp_path, enc, dtype):
    vol = source(dtype)
    p = str(tmp_path / ("v.mhd" if "data_file" in ENCODINGS[enc] else "v.mha"))
    surf.write_metaimage(p, vol, SPACING, ORIGIN, **ENCODINGS[enc])
    got, sp, org = surf.read_metaimage(p)
    assert got.dtype == vol.dtype and got.dtype.isnative
    assert np.array_equal(got.view(np.uint8), vol.view(np.uint8)) and sp == SPACING and org == ORIGIN


@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: np.dtype(d).name)
def test_element_byte_order_key_and_flips(built, tmp_path, dtype):
    """ElementByteOrderMSB means what BinaryDataByteOrderMSB does; the byte swap comes before the axis flips of a
    negative TransformMatrix diagonal, which move the origin as for native data."""
    vol = source(dtype, (4, 5, 6), seed=1)
    p = tmp_path / "e.mha"
    surf.write_metaimage(str(p), vol, SPACING, ORIGIN, byte_order=">", compress=6)
    p.write_bytes(p.read_bytes().replace(b"BinaryDataByteOrderMSB = True", b"ElementByteOrderMSB = True"))
    assert np.array_equal(surf.read_metaimage(str(p))[0], vol)
    flip = (-1, 0, 0, 0, 1, 0, 0, 0, -1)
    for kw in (dict(), dict(compress=6), dict(data_file="f.zraw", compress=1)):
        q = str(tmp_path / "f.mhd")
        surf.write_metaimage(q, vol, SPACING, ORIGIN, transform=flip, byte_order=">", **kw)
        plain = str(tmp_path / "plain.mha")
        surf.write_metaimage(plain, vol, SPACING, ORIGIN, transform=flip)
        got, sp, org = surf.read_metaimage(q)
        want = surf.read_metaimage(plain)
        assert np.array_equal(got, vol[::-1, :, ::-1]) and np.array_equal(got, want[0])
        assert org == want[2] == (ORIGIN[0] - SPACING[0] * 5, ORIGIN[1], ORIGIN[2] - SPACING[2] * 3)


def test_phases_reported(built, tmp_path):
    p = str(tmp_path / "t.mha")
    surf.write_metaimage(p, source(np.int16, (30, 40, 50)), compress=6, byte_order=">")
    ph = {}
    surf.read_metaimage(p, ph)
    assert sorted(ph) == ["header_s", "inflate_s", "read_s", "swap_s"] and all(v >= 0 for v in ph.values())
    assert ph["inflate_s"] > 0


# ---- refusals ---------------------------------------------------------------------------------------------------

def _compressed(tmp_path, **kw):
    vol = source(np.int16, (5, 6, 7), seed=2)
    p = tmp_path / "c.mha"
    surf.write_metaimage(str(p), vol, compress=6, **kw)
    return p, vol


def _header_end(raw):
    return raw.index(b"ElementDataFile = LOCAL\n") + len(b"ElementDataFile = LOCAL\n")


def refuse(path, *words):
    with pytest.raises(surf.FrogSurfError) as e:
        surf.read_metaimage(str(path))
    msg = str(e.value)
    for w in (str(path),) + words:
        assert w in msg, msg
    return msg


def test_truncated_stream(built, tmp_path):
    p, _ = _compressed(tmp_path, compressed_size=False)
    p.write_bytes(p.read_bytes()[:-40])
    refuse(p, "truncated")


def test_stream_shorter_than_dimsize(built, tmp_path):
    p, _ = _compressed(tmp_path)
    p.write_bytes(p.read_bytes().replace(b"DimSize = 7 6 5", b"DimSize = 7 6 6"))
    refuse(p, "ends after 420 of 504 bytes")


def test_stream_with_extra_output(built, tmp_path):
    p, _ = _compressed(tmp_path)
    p.write_bytes(p.read_bytes().replace(b"DimSize = 7 6 5", b"DimSize = 7 6 4"))
    refuse(p, "more than 336 bytes")


def test_corrupted_adler32(built, tmp_path):
    p, _ = _compressed(tmp_path)
    raw = bytearray(p.read_bytes())
    raw[-1] ^= 0x5A
    p.write_bytes(bytes(raw))
    refuse(p, "incorrect data check")


def test_corrupted_gzip_crc(built, tmp_path):
    p, _ = _compressed(tmp_path, gzip=True)
    raw = bytearray(p.read_bytes())
    raw[-6] ^= 0x01  # in the CRC-32 of the gzip trailer
    p.write_bytes(bytes(raw))
    refuse(p, "incorrect data check")


def test_bad_stream_header(built, tmp_path):
    p, _ = _compressed(tmp_path)
    raw = bytearray(p.read_bytes())
    raw[_header_end(bytes(raw))] = 0x00
    p.write_bytes(bytes(raw))
    refuse(p, "corrupt compressed stream")


def test_compressed_size_beyond_file(built, tmp_path):
    p, _ = _compressed(tmp_path)
    raw = p.read_bytes()
    n = len(raw) - _header_end(raw)
    p.write_bytes(raw.replace(b"CompressedDataSize = %d" % n, b"CompressedDataSize = %d" % (n + 1)))
    refuse(p, "CompressedDataSize = %d" % (n + 1), "exceeds")


def test_compressed_size_bounds_the_stream(built, tmp_path):
    """CompressedDataSize smaller than the stream: the stream is cut there."""
    p, _ = _compressed(tmp_path)
    raw = p.read_bytes()
    n = len(raw) - _header_end(raw)
    p.write_bytes(raw.replace(b"CompressedDataSize = %d" % n, b"CompressedDataSize = %d" % (n - 10)))
    refuse(p, "truncated")


def test_header_size_auto_with_compression(built, tmp_path):
    p = tmp_path / "a.mhd"
    surf.write_metaimage(str(p), source(np.int16), compress=6, data_file="a.zraw", header_size=-1)
    refuse(p, "HeaderSize = -1")


@pytest.mark.parametrize("old,new,words", [
    (b"ElementType = MET_SHORT", b"ElementType = MET_LONG", ["ElementType = MET_LONG", "platform"]),
    (b"ElementType = MET_SHORT", b"ElementType = MET_ULONG", ["ElementType = MET_ULONG", "platform"]),
    (b"ElementType = MET_SHORT", b"ElementType = MET_LONG_LONG", ["ElementType = MET_LONG_LONG", "2^53"]),
    (b"ElementType = MET_SHORT", b"ElementType = MET_ULONG_LONG", ["ElementType = MET_ULONG_LONG", "2^53"]),
    (b"ElementDataFile = LOCAL", b"ElementDataFile = LIST", ["ElementDataFile = LIST"]),
    (b"ElementDataFile = LOCAL", b"ElementDataFile = s%03d.raw 1 5 1", ["ElementDataFile = s%03d.raw 1 5 1"]),
    (b"BinaryData = True", b"BinaryData = False", ["BinaryData = False"]),
    (b"ElementType = MET_SHORT", b"ElementNumberOfChannels = 2\nElementType = MET_SHORT", ["ElementNumberOfChannels = 2"]),
], ids=["long", "ulong", "long_long", "ulong_long", "list", "pattern", "ascii", "two_channels"])
def test_refused_keys(built, tmp_path, old, new, words):
    p = tmp_path / "r.mha"
    surf.write_metaimage(str(p), source(np.int16))
    raw = p.read_bytes()
    assert old in raw
    p.write_bytes(raw.replace(old, new))
    refuse(p, *words)


def test_short_raw_data(built, tmp_path):
    p = tmp_path / "s.mhd"
    surf.write_metaimage(str(p), source(np.int16), data_file="s.raw", header_size=-1)
    raw = (tmp_path / "s.raw").read_bytes()
    (tmp_path / "s.raw").write_bytes(raw[-400:])
    refuse(p, "s.raw", "short data")


def test_surf3d_names_a_bad_stream(built, tmp_path):
    """bin/surf3d keeps its exit code 5 for an unreadable file and prints the reader's reason (no GPU needed: the
    volume is read before any CUDA call)."""
    p, _ = _compressed(tmp_path)
    raw = bytearray(p.read_bytes())
    raw[-1] ^= 0x5A
    p.write_bytes(bytes(raw))
    r = subprocess.run([build.SURF_BIN, str(p), "-o", str(tmp_path / "o")], capture_output=True, text=True)
    assert r.returncode == 5 and "Cannot load file" in r.stderr and "incorrect data check" in r.stderr
    assert not os.path.exists(tmp_path / "o.csv.gz")


def test_gzip_wrapper_is_a_gzip_member(tmp_path):
    """The writer's gzip option produces what gzip tools read (a check of the test writer itself)."""
    import gzip
    p = tmp_path / "g.mhd"
    vol = source(np.uint16)
    surf.write_metaimage(str(p), vol, compress=9, gzip=True, data_file="g.zraw")
    assert gzip.decompress((tmp_path / "g.zraw").read_bytes()) == vol.tobytes()
    surf.write_metaimage(str(p), vol, compress=9, data_file="g.zraw")
    assert zlib.decompress((tmp_path / "g.zraw").read_bytes()) == vol.tobytes()


def test_match_plans_mhd_and_compressed_entries(built, tmp_path):
    """bin/match counts .mhd entries and compressed volumes like .mha ones: by the voxels their header states."""
    vol = np.zeros((8, 8, 8), np.int16)
    entries = []
    for i, kw in enumerate([dict(), dict(data_file="a.zraw", compress=9), dict(compress=9), dict(data_file="b.raw")]):
        p = str(tmp_path / (f"v{i}.mhd" if "data_file" in kw else f"v{i}.mha"))
        surf.write_metaimage(p, vol, **kw)
        entries.append(p)
    (tmp_path / "l.txt").write_text("".join(e + "\n" for e in entries))
    r = subprocess.run([build.BIN, str(tmp_path / "l.txt"), "-plan", "1", "-surf3d", "-n 20000"], capture_output=True, text=True)
    assert r.returncode == 0 and "Planned GPUs : 1 (6 image pairs)" in r.stdout


def test_match_takes_mhd_as_volume(built, tmp_path):
    """A .mhd entry is a volume entry: without libfrogsurf.so beside bin/match it is refused as one (before any CUDA
    call), where a keypoint file would be parsed."""
    import shutil
    (tmp_path / "bin").mkdir()
    (tmp_path / "frog_b200").mkdir()
    shutil.copy(build.BIN, tmp_path / "bin" / "match")
    shutil.copy(build.LIB, tmp_path / "frog_b200" / "libfrogmatch.so")
    surf.write_metaimage(str(tmp_path / "v.mhd"), np.zeros((8, 8, 8), np.int16), data_file="v.zraw", compress=6)
    (tmp_path / "l.txt").write_text(str(tmp_path / "v.mhd") + "\n")
    env = {k: v for k, v in os.environ.items() if k != "LD_LIBRARY_PATH"}
    r = subprocess.run([str(tmp_path / "bin" / "match"), str(tmp_path / "l.txt")], capture_output=True, text=True, env=env)
    assert r.returncode == 1 and "MetaImage volumes (.mha / .mhd)" in r.stderr and "libfrogsurf.so" in r.stderr
