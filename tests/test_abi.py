"""CPU-side checks of the C ABI: the library loads without a GPU, exports every symbol include/thor_b200.h declares,
its work-item structs have the documented layout, and compute entry points fail loudly (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "thor_b200.h")


def header_symbols():
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    names = set()
    # per-sample macro block: expand ##SFX
    m = re.search(r"#define TB_DECL_SAMPLE_SYMBOLS\(S, SFX\)(.*?)(?=\n\nTB_DECL)", txt, flags=re.S)
    for fn in re.findall(r"(\w+)_##SFX\(", m.group(1)):
        names.update({fn + "_lbd", fn + "_hbd"})
    rest = txt.replace(m.group(0), "")
    rest = "\n".join(l for l in rest.splitlines() if not l.lstrip().startswith("#") and not l.startswith("TB_DECL"))
    for fn in re.findall(r"\b(\w+)\s*\([^;{}]*\)\s*;", rest):
        if not fn.startswith(("_", "TB_")):
            names.add(fn)
    for arr in re.findall(r"(coeffs_\w+)\[", rest):
        names.add(arr)
    return sorted(names)


def test_header_lists_the_reference_boundary():
    syms = header_symbols()
    # SURVEY.md §8b: the functions the reference's host objects import from the four kernel objects
    for base in ("sad_calc_simd", "ssd_calc_simd", "widesad_calc_simd", "sad_calc_fasthalf_simd", "sad_calc_fastquarter_simd", "detect_clpf_simd",
                 "detect_multi_clpf_simd", "block_avg_simd", "sad_calc_simd_unaligned", "clpf_block4", "clpf_block4_noclip", "clpf_block8",
                 "clpf_block8_noclip", "scale_frame_down2x2_simd", "get_inter_prediction_luma_simd", "get_inter_prediction_chroma_simd",
                 "cdef_find_dir_simd"):
        assert base + "_lbd" in syms and base + "_hbd" in syms
    for name in ("transform_simd", "inverse_transform_simd", "check_nz_area", "calc_cbp_simd", "cdef_filter_block_simd", "coeffs_standard_lbd",
                 "coeffs_bipred_hbd", "coeffs_chroma_lbd"):
        assert name in syms


def test_library_exports_every_declared_symbol():
    import thor_b200
    out = subprocess.run(["nm", "-D", "--defined-only", thor_b200.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if l.strip()}
    missing = [s for s in header_symbols() if s not in exported]
    assert not missing, missing


def test_reference_undefined_symbols_are_satisfied():
    """Every symbol the reference's HOST objects import from its kernel objects is defined by libthor_b200.so
    (checked against oracle/_ref/obj when the reference was built here)."""
    import thor_b200
    objdir = os.path.join(ROOT, "oracle", "_ref", "obj")
    if not os.path.isdir(objdir):
        pytest.skip("oracle/_ref not built")
    kernel_objs = {"enc/enc_kernels.o", "enc/enc_kernels_hbd.o", "common/common_kernels.o", "common/common_kernels_hbd.o"}
    defined_by_kernels, undefined_by_hosts = set(), set()
    for sub in ("enc", "common", "dec"):
        for f in os.listdir(os.path.join(objdir, sub)):
            rel = sub + "/" + f
            out = subprocess.run(["nm", os.path.join(objdir, rel)], capture_output=True, text=True, check=True).stdout
            for l in out.splitlines():
                parts = l.split()
                if rel in kernel_objs and len(parts) == 3 and parts[1] in "TDRB":
                    defined_by_kernels.add(parts[2])
                if rel not in kernel_objs and len(parts) == 2 and parts[0] == "U":
                    undefined_by_hosts.add(parts[1])
    needed = defined_by_kernels & undefined_by_hosts
    out = subprocess.run(["nm", "-D", "--defined-only", thor_b200.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if l.strip()}
    assert len(needed) >= 40
    assert not (needed - exported), sorted(needed - exported)


def test_struct_layouts_match_header(tmp_path):
    import thor_b200 as t
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "thor_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n",sizeof(tb_sad_item_t),'
                   'sizeof(tb_me_item_t),sizeof(tb_me_result_t),sizeof(tb_interp_item_t),sizeof(tb_txfm_item_t),sizeof(tb_txfm_result_t),'
                   'sizeof(tb_intra_item_t),sizeof(tb_blkinfo_t));printf("%zu %zu\\n",sizeof(tb_me_bi_item_t),sizeof(tb_combine_item_t));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    sizes = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [t.SAD_ITEM.itemsize, t.ME_ITEM.itemsize, t.ME_RESULT.itemsize, t.INTERP_ITEM.itemsize, t.TXFM_ITEM.itemsize,
                     t.TXFM_RESULT.itemsize, t.INTRA_ITEM.itemsize, t.BLKINFO.itemsize, t.ME_BI_ITEM.itemsize, t.COMBINE_ITEM.itemsize]


def test_no_cpu_fallback():
    """Without a CUDA device the library must refuse to compute (this test only asserts on GPU-less machines)."""
    import thor_b200 as t
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("GPU present")
    assert t.lib.tb_init(0) == t.TB_ERR_CUDA
    assert b"CUDA" in t.lib.tb_last_error()
    assert t.lib.tb_frame_create(64, 64, 32, 1) is None
    # the product never links the oracle
    out = subprocess.run(["ldd", t.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out and "thorref" not in out


def test_cpu_bench_driver_compiles_against_the_header():
    """oracle/cpu_bench.c shares the work-item structs of include/thor_b200.h: a field rename must not leave a stale prebuilt .so behind
    (build() recompiles it; this is the two-second version of that check)"""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run(["gcc", "-std=gnu99", "-fsyntax-only", "-w", os.path.join(root, "oracle", "cpu_bench.c")], capture_output=True, text=True, cwd=os.path.join(root, "oracle"))
    assert r.returncode == 0, r.stderr[-800:]


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "obj")), reason="oracle/_ref not built")
def test_binding_example_compiles_against_reference_headers():
    """examples/*.c (INTEGRATION.md §2.1 / §2.2 as real C) use the reference's own types (deblock_data_t, yuv_frame_t)
    and the C ABI header: the reference build (`make -C oracle ref`, -Wall -Werror) compiled them for both sample widths"""
    for src in ("frame_filters_binding", "motion_search_binding", "rdo_batch_server"):
        for width in ("lbd", "hbd"):
            obj = os.path.join(ROOT, "oracle", "_ref", "examples", "%s_%s.o" % (src, width))
            assert os.path.exists(obj), obj
            out = subprocess.run(["nm", "--defined-only", obj], capture_output=True, text=True, check=True).stdout
            assert out.strip(), "%s defines nothing" % obj


def test_rdo_struct_layouts_match_header(tmp_path):
    """tb_rdo_frame_t / tb_rdo_blk_t / tb_rdo_leaf_t (include/thor_b200.h) against their Python mirrors (thor_b200/rdo_jobs.py): sizes and the offsets of the
    fields the mirrors address; the RD-loop entry points are exported; without a GPU they refuse to compute."""
    import ctypes as C
    import thor_b200 as t
    from thor_b200 import rdo_jobs as RJ
    fields = ["width", "lambda", "early_skip_thr", "ref_sign", "orig", "orig_stride", "ref", "ref_stride", "ref_pad", "rec", "rec_stride", "blk", "leaves", "leaf_count", "coeffs"]
    src = tmp_path / "rdo.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "thor_b200.h"\nint main(){printf("%zu %zu %zu %d %d %d\\n",sizeof(tb_rdo_frame_t),sizeof(tb_rdo_blk_t),'
                   'sizeof(tb_rdo_leaf_t),TB_RDO_MAX_REF,TB_RDO_MAX_LEAVES,TB_RDO_SB_COEFFS);' +
                   "".join('printf("%%zu\\n",offsetof(tb_rdo_frame_t,%s));' % f for f in fields) +
                   'printf("%zu %zu %zu\\n",offsetof(tb_rdo_leaf_t,mv_arr0),offsetof(tb_rdo_leaf_t,coeff_ofs),offsetof(tb_rdo_leaf_t,cost));return 0;}\n')
    exe = tmp_path / "rdo"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert [int(v) for v in out[:6]] == [C.sizeof(RJ.RdoFrame), RJ.RDO_BLK.itemsize, RJ.RDO_LEAF.itemsize, RJ.TB_RDO_MAX_REF, RJ.TB_RDO_MAX_LEAVES, RJ.TB_RDO_SB_COEFFS]
    py = {"lambda": "lambda_"}
    assert [int(v) for v in out[6:6 + len(fields)]] == [getattr(RJ.RdoFrame, py.get(f, f)).offset for f in fields]
    assert [int(v) for v in out[6 + len(fields):]] == [RJ.RDO_LEAF.fields["mv_arr0"][1], RJ.RDO_LEAF.fields["coeff_ofs"][1], RJ.RDO_LEAF.fields["cost"][1]]
    for sym in ("tb_rdo_encode_frame", "tb_rdo_encode_frames", "tb_rdo_batch_create", "tb_rdo_batch_upload", "tb_rdo_batch_run", "tb_rdo_batch_download", "tb_rdo_batch_sync",
                "tb_rdo_batch_stats", "tb_rdo_batch_grid", "tb_rdo_batch_destroy", "tb_rdo_last_error", "tb_rdo_launch_count"):
        assert hasattr(t.lib, sym), sym
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if not has_gpu:  # no CPU path: the RD loop refuses without a device
        t.lib.tb_rdo_batch_create.restype = C.c_void_p
        assert t.lib.tb_rdo_batch_create(1, 1) is None
        f = RJ.RdoFrame()
        f.width, f.height, f.log2_sb_size, f.sample_bytes, f.bitdepth, f.qp = 64, 64, 7, 1, 8, 32
        dummy = (C.c_uint8 * 64)()
        f.blk = f.leaves = f.leaf_count = f.coeffs = C.addressof(dummy)
        assert t.lib.tb_rdo_encode_frame(C.byref(f)) == t.TB_ERR_CUDA
