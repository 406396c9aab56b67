"""SURVEY §8f.4: thor_b200/yuvio.py against the reference's own read_yuv_frame / write_yuv_frame (common/common_frame.c:478-654; their outputs
on seeded frames are stored in tests/golden/yuvio_reference.npz and, where oracle/_ref/libthorref.so is built, checked against a fresh call) and
its y4m header rules (enc/strings.c:376-449).  CPU only."""
import ctypes as C
import importlib.util
import io
import os

import numpy as np
import pytest

from _refstructs import Frame

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("yuvio", os.path.join(ROOT, "thor_b200", "yuvio.py"))
Y = importlib.util.module_from_spec(spec)
spec.loader.exec_module(Y)
REFSO = os.path.join(ROOT, "oracle", "_ref", "libthorref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden", "yuvio_reference.npz")
CASES = [(8, 8), (8, 10), (10, 10), (10, 8), (12, 10)]


def libc_file(path, mode):
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    fp = libc.fopen(path.encode(), mode.encode())
    assert fp
    return libc, fp


def make_input(directory, input_bd, bd):
    """a seeded 64x48 4:2:0 frame at input_bd bits in a file; returns (path, w, h, hbd)"""
    rng = np.random.default_rng(3 + input_bd * 16 + bd)
    w, h = 64, 48
    fdt = np.dtype("<u2") if input_bd > 8 else np.dtype("u1")
    path = os.path.join(directory, "in.yuv")
    with open(path, "wb") as f:
        for s in ((h, w), (h // 2, w // 2), (h // 2, w // 2)):
            f.write(rng.integers(0, 1 << input_bd, s).astype(fdt).tobytes())
    return path, w, h, int(max(input_bd, bd) > 8)


def reference_io(directory, input_bd, bd):
    """the compiled reference's read_yuv_frame of make_input's file, and its write_yuv_frame of the frame it read (None where the two are not
    comparable: when the file's depth is > 8 and differs from the codec's, the reference converts into `uint8_t *buf16` (common/common_frame.c:559,
    578-581), i.e. stores the low BYTE of every sample and writes uninitialised memory behind them)"""
    path, w, h, hbd = make_input(directory, input_bd, bd)
    ref = C.CDLL(REFSO)
    fr = Frame(w, h, bd, hbd)
    fr.s.input_bitdepth = input_bd
    libc, fp = libc_file(path, "rb")
    rd = ref.read_yuv_frame_hbd if hbd else ref.read_yuv_frame_lbd
    rd.argtypes = [C.c_void_p, C.c_void_p]
    rd(C.byref(fr.s), fp)
    libc.fclose(fp)
    planes = [fr.plane(p).copy() for p in range(3)]
    if input_bd > 8 and input_bd != bd:
        return planes, None
    out_ref = os.path.join(directory, "out_ref.yuv")
    libc, fp = libc_file(out_ref, "wb")
    wr = ref.write_yuv_frame_hbd if hbd else ref.write_yuv_frame_lbd
    wr.argtypes = [C.c_void_p, C.c_void_p]
    wr(C.byref(fr.s), fp)
    libc.fclose(fp)
    return planes, open(out_ref, "rb").read()


def golden(input_bd, bd):
    """what reference_io returned when the fixture was made (python tests/test_yuvio.py regenerates it)"""
    g, k = np.load(GOLDEN), "%d_%d" % (input_bd, bd)
    return [g["read_%s_%d" % (k, p)] for p in range(3)], (g["write_" + k].tobytes() if "write_" + k in g else None)


@pytest.mark.parametrize("input_bd,bd", CASES)
def test_read_and_write_match_reference(tmp_path, input_bd, bd):
    want, want_written = golden(input_bd, bd)
    if os.path.exists(REFSO):  # the fixture is what the reference computes today
        fresh, fresh_written = reference_io(str(tmp_path), input_bd, bd)
        assert all(np.array_equal(a, b) and a.dtype == b.dtype for a, b in zip(fresh, want)) and fresh_written == want_written, "fixture differs from the reference"
    path, w, h, hbd = make_input(str(tmp_path), input_bd, bd)
    with open(path, "rb") as f:
        got = Y.read_yuv_frame(f, w, h, input_bd, bd)
    for p in range(3):
        assert got[p].dtype == (np.uint16 if hbd else np.uint8)
        assert np.array_equal(got[p], want[p]), "read: plane %d differs" % p
    # the reference's writer on the frame it read; ours on the same samples
    if want_written is None:
        return
    buf = io.BytesIO()
    Y.write_yuv_frame(buf, got, input_bd, bd)
    assert buf.getvalue() == want_written, "write: bytes differ"


def test_y4m_header_and_reader(tmp_path):
    w, h, n = 32, 16, 3
    rng = np.random.default_rng(9)
    frames = [[rng.integers(0, 1024, s).astype("<u2") for s in ((h, w), (h // 2, w // 2), (h // 2, w // 2))] for _ in range(n)]
    path = str(tmp_path / "clip.y4m")
    with open(path, "wb") as f:
        f.write(b"YUV4MPEG2 W32 H16 F30000:1001 Ip A1:1 C420p10 XYSCSS=420P10\n")
        for fr in frames:
            f.write(b"FRAME\n")
            for p in fr:
                f.write(p.tobytes())
    hdr = Y.parse_y4m_header(open(path, "rb").read(256))
    assert (hdr.width, hdr.height, hdr.subsample, hdr.input_bitdepth, hdr.frame_headerlen) == (32, 16, 420, 10, 6)
    assert abs(hdr.frame_rate - 30000 / 1001) < 1e-9
    r = Y.YuvReader(path, skip=1)
    pinned_like = [np.zeros(p.shape, np.uint16) for p in frames[0]]     # caller-owned staging
    got = r.read(out=pinned_like)
    assert all(np.array_equal(got[p], frames[1][p]) and got[p] is pinned_like[p] for p in range(3))
    got = r.read()
    assert all(np.array_equal(got[p], frames[2][p]) for p in range(3))
    with pytest.raises(EOFError):
        r.read()
    r.close()
    assert Y.parse_y4m_header(b"\x00" * 64) is None
    with pytest.raises(ValueError):
        Y.parse_y4m_header(b"YUV4MPEG2 W32 H16 It C420\nFRAME\n")


if __name__ == "__main__":  # regenerate the fixture from the compiled reference (oracle/_ref)
    import tempfile
    store = {}
    for input_bd, bd in CASES:
        with tempfile.TemporaryDirectory() as tmp:
            planes, written = reference_io(tmp, input_bd, bd)
        k = "%d_%d" % (input_bd, bd)
        store.update({"read_%s_%d" % (k, p): a for p, a in enumerate(planes)})
        if written is not None:
            store["write_" + k] = np.frombuffer(written, np.uint8)
    np.savez_compressed(GOLDEN, **store)
    print(GOLDEN, sorted(store))
