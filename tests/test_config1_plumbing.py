"""BASELINE.json configs[0]: "Thordec single 64x64 I-frame bitstream on CPU -> bit-exact YUV (plumbing, no GPU)".  The reference's own CPU-runnable case: the compiled
reference encoder writes a one-I-frame 64x64 stream, the compiled reference decoder decodes it (both outputs stored as a fixture), and the decoded YUV — read back through thor_b200/yuvio.py (SURVEY §8f.4) —
equals the encoder's reconstruction sample for sample.  No GPU, no libthor_b200: this pins the container / file plumbing the GPU tests build on
(tests/test_dropin_link.py decodes the same kind of stream with Thordec_b200)."""
import importlib.util
import os
import subprocess

import numpy as np
import pytest

from test_dropin_link import HDB, REF, synth_yuv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("yuvio", os.path.join(ROOT, "thor_b200", "yuvio.py"))
Y = importlib.util.module_from_spec(spec)
spec.loader.exec_module(Y)
GOLDEN = os.path.join(ROOT, "tests", "golden", "config1_64x64.npz")
HAVE_REF = os.path.exists(os.path.join(REF, "Thorenc")) and os.path.exists(os.path.join(REF, "Thordec"))
W = H = 64


def reference_roundtrip(tmp, bitdepth):
    """the compiled reference encoder's reconstruction and the compiled reference decoder's output of its stream, as raw .yuv bytes"""
    synth_yuv(os.path.join(tmp, "in.yuv"), W, H, 1, bitdepth)
    extra = ["-bitdepth", str(bitdepth), "-input_bitdepth", str(bitdepth)] if bitdepth != 8 else []
    # tiny frames + CDEF corrupt the reference's frame header (SURVEY §8c.3): CDEF off
    r = subprocess.run([os.path.join(REF, "Thorenc")] + HDB + ["-cdef", "0", "-if", os.path.join(tmp, "in.yuv"), "-of", os.path.join(tmp, "a.bit"), "-rf", os.path.join(tmp, "rec.yuv"),
                                                              "-width", str(W), "-height", str(H), "-n", "1", "-qp", "32", "-f", "30"] + extra, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-800:]
    r = subprocess.run([os.path.join(REF, "Thordec"), os.path.join(tmp, "a.bit"), os.path.join(tmp, "dec.yuv")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-800:]
    return {k: open(os.path.join(tmp, k + ".yuv"), "rb").read() for k in ("rec", "dec")}


@pytest.mark.parametrize("bitdepth", [8, 10])
def test_single_64x64_intra_frame_roundtrip(tmp_path, bitdepth):
    """the reference's files are stored in tests/golden/config1_64x64.npz (python tests/test_config1_plumbing.py regenerates them); where the reference is
    built, a fresh round trip must reproduce them"""
    tmp = str(tmp_path)
    g = np.load(GOLDEN)
    files = {k: g["%s_%d" % (k, bitdepth)].tobytes() for k in ("rec", "dec")}
    if HAVE_REF:
        assert reference_roundtrip(tmp, bitdepth) == files, "the stored round trip differs from the reference's"
    else:
        synth_yuv(os.path.join(tmp, "in.yuv"), W, H, 1, bitdepth)
    for k, data in files.items():
        open(os.path.join(tmp, k + ".yuv"), "wb").write(data)
    w, h = W, H
    assert os.path.getsize(os.path.join(tmp, "dec.yuv")) == Y.frame_bytes(w, h, bitdepth)
    with open(os.path.join(tmp, "dec.yuv"), "rb") as fd, open(os.path.join(tmp, "rec.yuv"), "rb") as fr, open(os.path.join(tmp, "in.yuv"), "rb") as fi:
        dec = Y.read_yuv_frame(fd, w, h, bitdepth, bitdepth)
        rec = Y.read_yuv_frame(fr, w, h, bitdepth, bitdepth)
        src = Y.read_yuv_frame(fi, w, h, bitdepth, bitdepth)
    for p in range(3):
        assert np.array_equal(dec[p], rec[p]), "decoder output differs from the encoder's reconstruction (plane %d)" % p
    mse = float(np.mean((dec[0].astype(np.float64) - src[0].astype(np.float64)) ** 2)) / (1 << (2 * (bitdepth - 8)))
    assert mse < 40.0, "the decoded frame is not a coded version of the source (luma MSE %.1f at 8-bit scale)" % mse


if __name__ == "__main__":  # regenerate the fixture from the compiled reference (oracle/_ref)
    import tempfile
    store = {}
    for bd in (8, 10):
        with tempfile.TemporaryDirectory() as tmp:
            store.update({"%s_%d" % (k, bd): np.frombuffer(v, np.uint8) for k, v in reference_roundtrip(tmp, bd).items()})
    np.savez_compressed(GOLDEN, **store)
    print(GOLDEN, sorted(store))
