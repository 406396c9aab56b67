#!/usr/bin/env python
"""bench.py — Thor encode on B200: the RD loop of REAL encodes, in Mpixel/s (BASELINE.json metric: "encode Mpixels/s (1080p HDB_high_efficiency)").

WORKLOAD.  A synthetic 4:2:0 clip is encoded ONCE, untimed, by the unmodified reference encoder on the CPU (oracle/_ref/Thorenc_capture: the
reference's own objects + the observing shim).  The shim writes every frame's RD-loop JOB — the frame parameters the reference chose (type, qp,
lambda, reference list), the source planes and the padded RECONSTRUCTED reference frames of that real encode — together with what the reference's
process_block() decided for it (reconstruction before the in-loop filters, per-4x4 block state, RD cost per super block).  The jobs are the
workload; the reference's decisions are the expected answers.

ONE STEP = the RD loop (enc/encode_block.c:2401-2565 process_block over every super block: early skip, motion searches, RD candidates with
prediction -> DCT -> quant -> reconstruction -> SSD + bit count, intra, split decisions) of one steady-state GOP of the clip: the P frame and the 7 hierarchical B frames
of config_HDB_high_efficiency at 1920x1080 (the clip's only I frame is left out, in both arms) (--config selects the other BASELINE.json configurations).  That loop is 97 % of the reference
encoder's run time; the in-loop filters, the temporal interpolation and the bit writer are NOT in the step (both arms).  The frames of the GOP are
presented as independent jobs, as a server encoding several sequences (or intra-period segments) sees them: their inputs come from the capture,
so the inter-frame dependency of ONE sequence is not part of the measurement (tools/encode_bench.py times the sequential single-stream encode).
The K timed steps are K GOP replicas (distinct device buffers) submitted in ONE launch of the persistent kernel, which draws ready super blocks
from all of them — the wavefront of one frame is only ~4 super blocks wide, a GPU needs many frames in flight.

  value  frames resident in HBM, one launch, CUDA events on the launching stream
  e2e    tb_rdo_encode_frames-style: upload of every job from pinned host memory, launch, download of every decision (reconstruction, block
         state, leaf lists, coefficients), inside the timed region
  parity every frame of the LAST timed launch is compared with the reference's decisions (rec, block state, RD cost per super block): mismatch = exit 3

--impl reference / cpu_baseline: the reference encoder itself (Thorenc_capture) as one process per host thread, all encoding the full-size clip
continuously; throughput is read in fixed wall-clock slices (one slice = one step) from the progress the observing shim publishes per super block, in
the encoders' steady state (P + B frames), as pixels decided / seconds inside the reference's process_block loop (the RD loop the GPU arm times).

  python bench.py --gpus 1 --steps 5 --warmup 3
  python bench.py --impl reference --steps 1 --warmup 0
"""
import argparse
import ctypes as C
import hashlib
import importlib.util
import json
import os
import re
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(ROOT, "oracle", "_ref")

# the reference's configuration files (config_*.txt in the reference's root), as command-line flags of Thorenc
HDB = ("-HQperiod 1 -num_reorder_pics 7 -interp_ref 1 -dqpI -2 -dqpB0 3 -dqpB1 1 -dqpB2 0 -mqpP 1.2 -mqpB 1.2 -mqpB0 1.1 -mqpB1 1.2 -mqpB2 1.3 "
       "-lambda_coeffI 0.8 -lambda_coeffP 1.2 -lambda_coeffB 1.2 -lambda_coeffB0 1.2 -lambda_coeffB1 1.2 -lambda_coeffB2 1.2 -intra_rdo 1 -enable_tb_split 1 "
       "-enable_pb_split 1 -early_skip_thr 0.3 -max_num_ref 4 -use_block_contexts 1 -enable_bipred 1 -encoder_speed 0 -enable_cfl_intra 1 -enable_cfl_inter 0")
HDB16 = ("-HQperiod 1 -num_reorder_pics 15 -interp_ref 1 -dqpI -2 -dqpB0 2 -dqpB1 1 -dqpB2 0 -dqpB3 0 -mqpP 1.2 -mqpB 1.2 -mqpB0 1.075 -mqpB1 1.15 -mqpB2 1.225 -mqpB3 1.3 "
         "-lambda_coeffI 0.8 -lambda_coeffP 1.2 -lambda_coeffB 1.2 -lambda_coeffB0 1.2 -lambda_coeffB1 1.2 -lambda_coeffB2 1.2 -lambda_coeffB3 1.2 -intra_rdo 1 "
         "-enable_tb_split 1 -enable_pb_split 1 -early_skip_thr 0.3 -max_num_ref 4 -use_block_contexts 1 -enable_bipred 1 -encoder_speed 0 -enable_cfl_intra 1 "
         "-enable_cfl_inter 0")
LDB = ("-HQperiod 12 -mqpP 1.2 -dqpI -2 -lambda_coeffI 0.8 -lambda_coeffP 1.2 -intra_rdo 0 -enable_tb_split 0 -enable_pb_split 0 -early_skip_thr 1.0 "
       "-max_num_ref 2 -use_block_contexts 1 -enable_bipred 0 -encoder_speed 2 -enable_cfl_intra 1 -enable_cfl_inter 0 -cdef 0 -clpf 1")
CONFIGS = {
    #         W     H     bitdepth frames flags                         reference config file
    "hdb":   (1920, 1080, 8,  9,  HDB,                          "config_HDB_high_efficiency"),     # BASELINE.json configs[2]: the headline
    "ldb":   (1920, 1080, 8,  9,  LDB,                          "config_LDB_low_complexity"),      # configs[1]
    "ra4k":  (3840, 2160, 8,  9,  HDB + " -intra_period 64",    "config_RA_high_efficiency"),      # configs[3]
    "hdb10": (1920, 1080, 10, 17, HDB16,                        "config_HDB16_high_efficiency"),   # configs[4]
}
QP = 32


class Cfg:
    def __init__(self, name, size=None, frames=None):
        self.name = name
        self.W, self.H, self.BD, self.frames, flags, self.cfgfile = CONFIGS[name]
        if size:
            self.W, self.H = size
        if frames:
            self.frames = frames
        self.flags = flags.split()
        self.ESZ = 1 if self.BD == 8 else 2

    def enc_flags(self, w, h, n):
        f = list(self.flags) + ["-width", str(w), "-height", str(h), "-n", str(n), "-qp", str(QP), "-f", "30"]
        if self.BD != 8:
            f += ["-bitdepth", str(self.BD), "-input_bitdepth", str(self.BD)]
        return f

    def workload(self):
        return ("RD loop (process_block over every super block) of the %d inter frames (one steady-state GOP) of a real %dx%d %d-bit 4:2:0 %s encode (qp %d) per "
                "step; jobs = frame parameters + source + reconstructed references captured from the reference encoder; frames presented as independent jobs; "
                "in-loop filters, temporal interpolation and bit writer not included" % (self.frames - 1, self.W, self.H, self.BD, self.cfgfile.replace("config_", ""), QP))

    def metric(self):
        return "encode Mpixels/s (%dp %s, RD loop of real encodes)" % (self.H, self.cfgfile.replace("config_", ""))


# ----------------------------------------------------------------------------------------------------------------------
# the clip and its capture (setup, untimed)
# ----------------------------------------------------------------------------------------------------------------------
def synth_clip(path, w, h, n, bitdepth, seed=5, x0=0, y0=0, full=None):
    """moving 8x8-block texture + low-frequency sinusoids + N(0,2) noise, 4:2:0 (SURVEY.md §8d synthetic input).  A window (x0, y0, w, h) of the
    full-size clip `full` = (W, H) has the same samples as that region of the full clip."""
    W, H = full or (w, h)
    rng = np.random.default_rng(seed)
    m = 2 * n + 8
    yy, xx = np.mgrid[0:H + m, 0:W + m]
    base = np.clip(rng.integers(0, 48, ((H + m) // 8 + 1, (W + m) // 8 + 1)).repeat(8, 0).repeat(8, 1)[:H + m, :W + m] + 60 * np.sin(xx / 17.0) + 50 * np.cos(yy / 11.0) + 100,
                   0, 255)
    with open(path, "wb") as f:
        for k in range(n):
            y = np.clip(base[k:k + H, 2 * k:2 * k + W] + rng.normal(0, 2, (H, W)), 0, 255).astype(np.uint8)
            u = np.clip(128 + 20 * np.sin(xx[:H // 2, :W // 2] / 9.0 + k), 0, 255).astype(np.uint8)
            v = np.clip(128 + 20 * np.cos(yy[:H // 2, :W // 2] / 7.0), 0, 255).astype(np.uint8)
            lo = [rng.integers(0, 1 << (bitdepth - 8), p.shape).astype(np.uint16) for p in (y, u, v)] if bitdepth != 8 else None
            for i, p in enumerate((y, u, v)):
                s = 1 if i == 0 else 2
                if bitdepth != 8:
                    p = ((p.astype(np.uint16) << (bitdepth - 8)) | lo[i]).astype("<u2")
                f.write(np.ascontiguousarray(p[y0 // s:(y0 + h) // s, x0 // s:(x0 + w) // s]).tobytes())


def need(exe):
    p = os.path.join(REF, exe)
    if not os.path.exists(p):
        raise SystemExit("%s is missing: build it in the development container (python -c 'import __graft_entry__ as g; g.build()'); it travels with the repo" % p)
    return p


def capture_jobs(cfg, cache_root):
    """encode the clip once with the reference encoder + observing shim; returns (job directory, meta)"""
    key = hashlib.sha1(("%s %d %d %d %d %s v3" % (cfg.name, cfg.W, cfg.H, cfg.BD, cfg.frames, " ".join(cfg.flags))).encode()).hexdigest()[:12]
    d = os.path.join(cache_root, "%s_%dx%d_%d_%s" % (cfg.name, cfg.W, cfg.H, cfg.frames, key))
    meta_path = os.path.join(d, "meta.json")
    if os.path.exists(meta_path):
        return d, json.load(open(meta_path))
    shutil.rmtree(d, ignore_errors=True)
    os.makedirs(d)
    clip = os.path.join(d, "in.yuv")
    synth_clip(clip, cfg.W, cfg.H, cfg.frames, cfg.BD)
    t = time.time()
    r = subprocess.run([need("Thorenc_capture")] + cfg.enc_flags(cfg.W, cfg.H, cfg.frames) + ["-if", clip, "-of", os.path.join(d, "ref.bit"), "-rf", os.path.join(d, "ref_rec.yuv")],
                       capture_output=True, text=True, env=dict(os.environ, TB_RDO_DUMP=d, TB_RDO_STATS="1"))
    wall = time.time() - t
    m = re.search(r"in the reference's process_block ([\d.]+)", r.stderr)
    if r.returncode != 0 or not m:
        raise SystemExit("capture encode failed: %s" % (r.stderr[-1500:],))
    os.remove(clip); os.remove(os.path.join(d, "ref_rec.yuv"))
    meta = {"capture_wall_s": round(wall, 2), "reference_rd_loop_s": float(m.group(1)), "frames": cfg.frames, "pixels": cfg.W * cfg.H * cfg.frames,
            "reference_1thread_rd_loop_mpixel_s": round(cfg.W * cfg.H * cfg.frames / float(m.group(1)) / 1e6, 4),
            "reference_1thread_whole_encoder_mpixel_s": round(cfg.W * cfg.H * cfg.frames / wall / 1e6, 4)}
    json.dump(meta, open(meta_path, "w"))
    return d, meta


# ----------------------------------------------------------------------------------------------------------------------
# clocks sampling
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML from a thread every 5 ms (nvidia-smi -lms as fallback)."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index=0):
        self.sm, self.mx, self.reasons, self.index = [], [], set(), index
        self.proc, self.thread, self.stop_flag, self.nvml = None, None, threading.Event(), None

    def _nvml_loop(self):
        import pynvml as nv
        h = self.nvml
        while not self.stop_flag.is_set():
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                for bit, name in self.REASONS:
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else self.index
            self.nvml = nv.nvmlDeviceGetHandleByIndex(phys)
            self.mx.append(int(nv.nvmlDeviceGetMaxClockInfo(self.nvml, nv.NVML_CLOCK_SM)))
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True); self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                                          "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._smi_read, daemon=True); self.thread.start()
        except Exception:
            self.proc = None

    def _smi_read(self):
        names = [n for _, n in self.REASONS]
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            if r and r[0].isdigit():
                self.sm.append(int(r[0]))
            if len(r) > 1 and r[1].isdigit():
                self.mx.append(int(r[1]))
            for i in range(4):
                if len(r) >= 6 and r[2 + i].lower().startswith("active"):
                    self.reasons.add(names[i])

    def stop(self):
        self.stop_flag.set()
        if self.proc:
            self.proc.terminate()
        if self.thread:
            self.thread.join(timeout=1.0)
        return {"sm_mhz": int(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def load_rdo_jobs_module():
    """thor_b200/rdo_jobs.py without importing the package (the package dlopens libthor_b200.so; the CPU arm must not)"""
    spec = importlib.util.spec_from_file_location("thor_b200_rdo_jobs", os.path.join(ROOT, "thor_b200", "rdo_jobs.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


STAT_NAMES = ["cyc_interp", "cyc_me", "cyc_me_bi", "cyc_tx_chain", "cyc_coeff_bits", "cyc_ssd_sad", "cyc_intra", "cyc_copy", "cyc_early_skip", "cyc_idle", "cyc_total",
              "searches", "int_block_sads", "subpel_probes", "search_samples", "predictions", "prediction_samples", "txfm_chains", "txfm_samples", "intra_predictions",
              "intra_samples", "ssd_sad_samples", "super_blocks"] + ["cyc_me_%d" % (8 << k) for k in range(5)] + ["cyc_tx_%d" % (4 << k) for k in range(6)] + \
             ["cyc_ip_%d" % (4 << k) for k in range(6)] + ["ph_" + n for n in ("other", "early_skip", "skip_merge_cand", "search", "inter_cand", "bipred", "intra_search", "intra_cand",
                                                                               "commit")] + ["me_stage_" + n for n in ("telescope", "candidates", "hexagon", "halfpel", "quarterpel")]


DUMP_ARRAY_BYTES = 7_500_000  # per array; eight arrays stay under 64 MB in all


def dump_outputs(directory, frames):
    """--dump-outputs: what tb_rdo_encode_frames returns for the given frames (one GOP), as DIR/<name>.npy for comparing two builds output for
    output.  Samples become float32, wider integers float64 (both exact).  An array above DUMP_ARRAY_BYTES is replaced by a fixed, seeded sample of
    its elements (1-D) or rows (2-D): the same positions in every run with the same arguments."""
    def save(name, a, dtype):
        a = np.ascontiguousarray(a, dtype=dtype)
        row = a[0].nbytes if a.ndim > 1 and len(a) else a.itemsize
        n = max(1, DUMP_ARRAY_BYTES // row)
        if len(a) > n:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), n, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)

    os.makedirs(directory, exist_ok=True)
    blk_fields = [n for n in frames[0].blk.dtype.names if n != "pad"]
    leaf_cols = lambda lv: np.concatenate([lv[n].reshape(len(lv), -1).astype(np.float64) for n in lv.dtype.names], axis=1)
    count = lambda size, split: (4 if split else 1) * min(size // 2 if split else size, 16) ** 2  # coeff_count() of thor_b200/csrc/tb_rdo.h
    leaves, coeffs = [], []
    for hf in frames:
        for s in range(hf.job.nsb):
            lv = hf.leaves[s, :hf.leaf_count[s]]
            leaves.append(leaf_cols(lv))
            for size, split, ofs in zip(lv["size"].astype(int), lv["tb_split"].astype(int), lv["coeff_ofs"].astype(int)):
                if ofs >= 0:  # a coded block's coefficients: luma, then the two chroma runs; the rest of the area is not written
                    n = count(size, split) + 2 * count(size // 2, split and size // 2 > 4)
                    coeffs.append(hf.coeffs[s, ofs:ofs + n])
    for p, name in enumerate(("rec_y", "rec_u", "rec_v")):
        save(name, np.concatenate([hf.rec[p].reshape(-1) for hf in frames]), np.float32)
    save("blk", np.concatenate([np.stack([hf.blk[n].astype(np.float32) for n in blk_fields], axis=1) for hf in frames]), np.float32)
    save("leaf_count", np.concatenate([hf.leaf_count for hf in frames]), np.float64)
    save("sb_cost", np.concatenate([[hf.leaves["cost"][s, :hf.leaf_count[s]].astype(np.int64).sum() for s in range(hf.job.nsb)] for hf in frames]), np.float64)
    save("leaves", np.concatenate(leaves), np.float64)
    save("coeffs", np.concatenate(coeffs) if coeffs else np.zeros(0, np.int16), np.float32)


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
def run_gpu(args, cfg):
    import torch
    import torch.distributed as dist
    import thor_b200 as tb
    from thor_b200 import rdo_jobs as RJ

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    tb.init(local)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    tb.check(tb.lib.tb_set_stream(C.c_void_p(stream.cuda_stream)))
    L = tb.lib
    L.tb_rdo_batch_create.restype = C.c_void_p
    L.tb_rdo_batch_create.argtypes = [C.c_int, C.c_int]
    L.tb_rdo_batch_upload.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.tb_rdo_batch_run.argtypes = [C.c_void_p, C.c_int]
    L.tb_rdo_batch_download.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.tb_rdo_batch_sync.argtypes = [C.c_void_p]
    L.tb_rdo_batch_grid.argtypes = [C.c_void_p]
    L.tb_rdo_batch_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.tb_rdo_batch_destroy.argtypes = [C.c_void_p]
    L.tb_rdo_last_error.restype = C.c_char_p
    L.tb_rdo_launch_count.restype = C.c_uint64

    def ck(rc, what):
        if rc != 0:
            raise SystemExit("%s failed (%d): %s" % (what, rc, L.tb_rdo_last_error().decode()))

    # ---- workload (rank 0 captures; the cache directory is shared by the ranks of the node)
    if rank == 0:
        jobdir, meta = capture_jobs(cfg, args.cache)
    if world > 1:
        dist.barrier()
    if rank != 0:
        jobdir, meta = capture_jobs(cfg, args.cache)
    jobs = [j for j in RJ.load_jobs(jobdir) if j.hdr.frame_type != 0]  # steady state: the clip's I frame is not part of the step (both arms)
    nfr = len(jobs)
    gop_pixels = sum(j.pixels for j in jobs)
    K, Wm = args.steps, args.warmup
    nslots = nfr * max(K, Wm)
    alloc = lambda n: L.tb_malloc_host(max(n, 16))
    base = [RJ.HostFrame(j, alloc) for j in jobs]                       # replica 0: owns the pinned inputs
    hosts = base + [RJ.HostFrame(jobs[i % nfr], alloc, share_inputs=base[i % nfr]) for i in range(nfr, nslots)]  # replicas: own outputs, shared inputs
    batch = L.tb_rdo_batch_create(nslots, cfg.ESZ)
    if not batch:
        raise SystemExit("tb_rdo_batch_create: %s" % L.tb_rdo_last_error().decode())
    h2d = sum(j.in_bytes() for j in jobs); d2h = sum(j.out_bytes() for j in jobs)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def upload(n):
        for s in range(n):
            ck(L.tb_rdo_batch_upload(batch, s, C.byref(hosts[s].desc)), "tb_rdo_batch_upload")

    def download(n):
        for s in range(n):
            ck(L.tb_rdo_batch_download(batch, s, C.byref(hosts[s].desc)), "tb_rdo_batch_download")

    ev = lambda: torch.cuda.Event(enable_timing=True)
    launches0 = int(L.tb_rdo_launch_count())
    # ---- resident frames; warm-up launch (W GOPs), then the timed launch (K GOPs)
    upload(nslots)
    barrier()
    if Wm > 0:
        ck(L.tb_rdo_batch_run(batch, nfr * Wm), "tb_rdo_batch_run"); ck(L.tb_rdo_batch_sync(batch), "warm-up launch")
    sampler = ClockSampler(local); sampler.start()
    barrier()
    e0, e1 = ev(), ev()
    e0.record(stream)
    ck(L.tb_rdo_batch_run(batch, nfr * K), "tb_rdo_batch_run")
    e1.record(stream)
    ck(L.tb_rdo_batch_sync(batch), "timed launch")
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:  # the decisions of the last timed step (its GOP replica), downloaded after the timed region
        download_last = range(nfr * (K - 1), nfr * K)
        for s in download_last:
            ck(L.tb_rdo_batch_download(batch, s, C.byref(hosts[s].desc)), "tb_rdo_batch_download")
        ck(L.tb_rdo_batch_sync(batch), "download of the last step")
        dump_outputs(args.dump_outputs, [hosts[s] for s in download_last])
    stats = (C.c_uint64 * len(STAT_NAMES))()
    L.tb_rdo_batch_stats(batch, stats, len(STAT_NAMES))
    st = dict(zip(STAT_NAMES, [int(v) for v in stats]))
    grid = int(L.tb_rdo_batch_grid(batch))

    # ---- end to end: pinned host -> HBM, launch, decisions -> pinned host, every step's frames, inside the timed region.
    # N > 1: the data plane north_star names — rank 0 owns the raw source frames of every rank's GOP, uploads and scatters them over NCCL; every rank
    # returns its RD costs per super block by an NCCL gather
    for hf in hosts:
        hf.clear_outputs()
    Ke = min(K, args.e2e_steps) if args.e2e_steps > 0 else K
    coll_ms = 0.0
    scatter_bytes = gather_bytes = 0
    if world > 1:
        src_elems = sum(p.size for j in jobs for p in j.orig)
        tdt = torch.uint8 if cfg.ESZ == 1 else torch.int16
        mine_src = torch.empty(src_elems, dtype=tdt, device="cuda")
        if rank == 0:
            flat = np.concatenate([p.reshape(-1) for j in jobs for p in j.orig])
            pin = torch.from_numpy(flat.view(np.uint8 if cfg.ESZ == 1 else np.int16).copy()).pin_memory()
        cost_dev = torch.zeros(sum(j.nsb for j in jobs), dtype=torch.int32, device="cuda")
        scatter_bytes = (world - 1) * src_elems * cfg.ESZ; gather_bytes = (world - 1) * cost_dev.numel() * 4
        # untimed warm-up of the two collectives (NCCL sets its point-to-point connections up on first use)
        if rank == 0:
            dist.scatter(mine_src, [pin.to("cuda", non_blocking=True) for _ in range(world)], src=0)
            dist.gather(cost_dev, [torch.empty_like(cost_dev) for _ in range(world)], dst=0)
        else:
            dist.scatter(mine_src, None, src=0)
            dist.gather(cost_dev, None, dst=0)
    barrier()
    t0, t1 = ev(), ev()
    c0, c1, c2, c3 = ev(), ev(), ev(), ev()
    t0.record(stream)
    if world > 1:
        c0.record(stream)
        if rank == 0:
            src_list = [pin.to("cuda", non_blocking=True) for _ in range(world)]  # one upload per rank's GOP (the ranks encode the same clip)
            dist.scatter(mine_src, src_list, src=0)
        else:
            dist.scatter(mine_src, None, src=0)
        c1.record(stream)
        # the scattered source planes replace the host source pointers of replica 0 of every frame (device pointers: the copies are cudaMemcpyDefault)
        o = 0
        for i, j in enumerate(jobs):
            for p in range(3):
                hosts[i].desc.orig[p] = mine_src.data_ptr() + o * cfg.ESZ
                o += j.orig[p].size
    upload(nfr * Ke)
    ck(L.tb_rdo_batch_run(batch, nfr * Ke), "tb_rdo_batch_run")
    download(nfr * Ke)
    if world > 1:
        c2.record(stream)
        glist = [torch.empty_like(cost_dev) for _ in range(world)] if rank == 0 else None
        dist.gather(cost_dev, glist, dst=0)
        c3.record(stream)
    t1.record(stream)
    ck(L.tb_rdo_batch_sync(batch), "end-to-end launch")
    barrier()
    ems = t0.elapsed_time(t1)
    if world > 1:
        coll_ms = c0.elapsed_time(c1) + c2.elapsed_time(c3)
    clocks = sampler.stop()
    launches = int(L.tb_rdo_launch_count()) - launches0

    # ---- parity: every frame of the end-to-end launch against the reference's decisions
    par = {"rec": 0, "blk": 0, "sb_cost": 0}
    for s in range(nfr * Ke):
        r = hosts[s].check()
        for k in par:
            par[k] += int(r[k])
    nchk = nfr * Ke
    parity_ok = all(v == nchk for v in par.values())

    if world > 1:
        t = torch.tensor([ms, ems, coll_ms, 0.0 if parity_ok else 1.0], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ems, coll_ms, bad = [float(v) for v in t.tolist()]
        parity_ok = bad == 0.0
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    value = world * K * gop_pixels / (ms * 1e-3) / 1e6
    e2e_value = world * Ke * gop_pixels / (ems * 1e-3) / 1e6
    alg_samples = st["search_samples"] + st["prediction_samples"] + st["txfm_samples"] + st["intra_samples"] + st["ssd_sad_samples"]
    alg_bytes = alg_samples * cfg.ESZ
    achieved = alg_bytes / (ms * 1e-3) / 1e9
    busy = 1.0 - st["cyc_idle"] / max(1, st["cyc_total"])
    tr = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[cfg.name]["rdo_batch_kernel"]
    except Exception:
        pass
    S = "uint8_t" if cfg.ESZ == 1 else "uint16_t"
    line = {
        "metric": cfg.metric(), "value": round(value, 4), "unit": "Mpixel/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms / K, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8" if cfg.ESZ == 1 else "u16", "data": "synthetic",
        "config": {"workload": cfg.workload(), "frames_per_step": nfr, "steps_in_one_launch": K, "ctas": grid,
                   "parallelism": ("GOP-per-GPU x%d; rank 0 scatters the raw source frames over NCCL and gathers one int32 per super block from every rank (stand-in payload of the size of the RD costs; the decisions themselves are downloaded to each rank's host)" % world) if world > 1 else "1 GPU, no collective",
                   "l2_policy": "per-launch inputs+outputs %.0f MB > 126 MB L2" % ((h2d + d2h) * K / 1e6)},
        "e2e": {"value": round(e2e_value, 4), "unit": "Mpixel/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": round(ems / Ke, 2), "steps": Ke},
        "gpu_launches": launches,
        "clocks": clocks,
        "parity": {"frames_checked": nchk, "rec_equal": par["rec"], "block_state_equal": par["blk"], "sb_cost_equal": par["sb_cost"], "ok": parity_ok,
                   "checker": "reference (process_block of the compiled reference encoder, captured with the jobs)"},
        "roofline": {"kernel": "rdo_batch_kernel<%s> (the whole RD loop: a1-a16 primitives under the process_block control flow)" % S,
                     # contract fields: ALGORITHMIC bytes (SURVEY.md §8d per-unit figures x the units the data-dependent loop actually executed, counted by the kernel)
                     # / launch time vs the measured HBM peak.  The kernel is NOT HBM-bound: it is a dependency chain (serial block decisions inside a super
                     # block, wavefront between super blocks); what bounds it is single-warp latency, see `binding`
                     "bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                     "unit": "GB/s", "frac": round(achieved / peak, 5),
                     # DRAM bytes of this launch, scaled per super block from the committed ncu capture of the same kernel on a smaller batch (profiles/ncu_traffic.json)
                     "traffic": int(tr["dram_bytes_total"] / tr["super_blocks"] * st["super_blocks"]) if tr and tr.get("super_blocks") else None,
                     "traffic_source": tr.get("capture") if tr else None,
                     "binding": "instruction delivery (ncu: ~19 stalled warps per issued instruction wait for instructions; issue slots 4 % busy; DRAM 0.1 %, L2 2 % of peak): "
                                "a serial decision chain per super block run by one 8-warp CTA whose code streams from L2",
                     "cta_busy_frac": round(busy, 4), "algorithmic_bytes": int(alg_bytes), "ms_per_launch": round(ms, 2), "share_of_step": 1.0,
                     "ncu": {k: tr[k] for k in tr if k.endswith("_pct") or k.startswith("stalled_")} if tr else None,
                     "work": {k: st[k] for k in STAT_NAMES[11:23]},
                     "cycles_share": {k[4:]: round(st[k] / max(1, st["cyc_total"]), 4) for k in STAT_NAMES[:10] + STAT_NAMES[23:40]},
                     "phase_share_of_a_super_block": {k[3:]: round(st[k] / max(1, sum(st[n] for n in STAT_NAMES[40:49])), 4) for k in STAT_NAMES[40:49]},
                     "small_search_stage_share": {k[9:]: round(st[k] / max(1, sum(st[n] for n in STAT_NAMES[49:54])), 4) for k in STAT_NAMES[49:54]}},
        "single_stream_reference": meta,
    }
    if world > 1:
        line["collective"] = {"backend": "nccl", "scatter_bytes_per_step": int(scatter_bytes // max(1, Ke)), "gather_bytes_per_step": int(gather_bytes // max(1, Ke)),
                              "ms": round(coll_ms, 3), "share_of_e2e": round(coll_ms / ems, 5)}
    if not args.no_cpu and world == 1:  # the reported CPU baseline is measured at N = 1 only
        line["cpu_baseline"] = cpu_arm(args, cfg, brief=True)
    print(json.dumps(line))
    L.tb_rdo_batch_destroy(batch)
    if not parity_ok:
        sys.stderr.write("PARITY FAILURE: the device's decisions differ from the reference's on the bench jobs: %s of %d frames\n" % (par, nchk))
        sys.exit(3)


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference encoder itself, one process per host thread
# ----------------------------------------------------------------------------------------------------------------------
def cpu_arm(args, cfg, brief=False):
    """One unmodified reference encoder per host thread, all encoding the full-size clip (2 GOPs + 1 frames) continuously.  After every process has
    passed its I and first P frame (steady state: P + hierarchical B frames), throughput is measured in fixed wall-clock SLICES (= steps) from the
    progress the observing shim publishes after every super block (TB_RDO_PROGRESS: pixels decided, seconds inside process_block); the encoders are
    stopped after the last slice.  value = mean over timed slices of sum over processes of (pixels decided in the slice / seconds spent inside
    process_block in the slice): the RD loop only, the quantity the GPU arm times."""
    import struct
    cores = len(os.sched_getaffinity(0))
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
    except Exception:
        phys = None
    nproc = args.cpu_procs or cores
    if brief and not args.cpu_fresh:  # cpu_baseline of the GPU arm: a measurement of this box less than an hour old (the --impl reference run) is reused
        try:
            for d in sorted(os.listdir(args.cache)):
                if d.startswith("cpu_arm_%s_%dx%d_" % (cfg.name, cfg.W, cfg.H)):
                    last = json.load(open(os.path.join(args.cache, d, "last_result.json")))
                    if time.time() - last["time"] < 3600 and last["res"]["cores"] == nproc:
                        last["res"]["reused"] = "measured %.0f s earlier on this box by bench.py --impl reference / a previous run (--cpu-fresh re-measures)" % (time.time() - last["time"])
                        return last["res"]
        except Exception:
            pass
    gop = 1
    if "-num_reorder_pics" in cfg.flags:
        gop = int(cfg.flags[cfg.flags.index("-num_reorder_pics") + 1]) + 1
    nfr = max(17, 2 * gop + 1)
    tmp = os.path.join(args.cache, "cpu_arm_%s_%dx%d_%d" % (cfg.name, cfg.W, cfg.H, nfr))
    os.makedirs(tmp, exist_ok=True)
    clip = os.path.join(tmp, "in.yuv")
    if not os.path.exists(clip):
        synth_clip(clip + ".tmp", cfg.W, cfg.H, nfr, cfg.BD)
        os.replace(clip + ".tmp", clip)
    exe = need("Thorenc_capture")
    reference = args.impl == "reference"
    n_warm = args.warmup if reference else 1
    n_timed = max(1, args.steps) if reference else args.cpu_slices
    slice_s = args.cpu_slice if args.cpu_slice > 0 else min(4.0, max(1.5, 60.0 / (n_warm + n_timed)))
    prog = [os.path.join(tmp, "progress_%d" % i) for i in range(nproc)]
    for f in prog:
        if os.path.exists(f):
            os.remove(f)
    ps = [subprocess.Popen([exe] + cfg.enc_flags(cfg.W, cfg.H, nfr) + ["-if", clip, "-of", os.path.join(tmp, "o%d.bit" % i)], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, TB_RDO_PROGRESS=prog[i])) for i in range(nproc)]

    tick = os.sysconf("SC_CLK_TCK")

    def cpu_seconds():  # CPU time the encoders have consumed so far (utime + stime of /proc/<pid>/stat)
        tot = 0.0
        for p in ps:
            try:
                f = open("/proc/%d/stat" % p.pid).read().rsplit(")", 1)[1].split()
                tot += (int(f[11]) + int(f[12])) / tick
            except Exception:
                pass
        return tot

    def read():
        out = []
        for f in prog:
            try:
                out.append(struct.unpack("<QdQ", open(f, "rb").read(24)))
            except Exception:
                out.append((0, 0.0, 0))
        return out

    slices, early = [], False
    try:
        t_start = time.time()
        settle_frames = 2 if gop > 1 else 1
        while True:  # steady state: every encoder is past its I (and first P) frame
            st = read()
            if all(s[2] >= settle_frames for s in st):
                break
            if any(p.poll() is not None for p in ps) or time.time() - t_start > args.cpu_settle_limit:
                early = True
                break
            time.sleep(0.25)
        settle_s = time.time() - t_start
        prev, t_prev = read(), time.time()
        cpu_prev, cpu_used, cpu_wall = cpu_seconds(), 0.0, 0.0
        for k in range(n_warm + n_timed):
            if early:
                break
            time.sleep(max(0.0, t_prev + slice_s - time.time()))
            cur, t_cur = read(), time.time()
            if any(p.poll() is not None for p in ps):
                early = True  # an encoder finished its clip (development sizes): the slice is not a steady-state sample
                break
            cpu_cur = cpu_seconds()
            if k >= n_warm:
                rd = sum((c[0] - a[0]) / (c[1] - a[1]) for a, c in zip(prev, cur) if c[1] > a[1]) / 1e6
                wall = sum(c[0] - a[0] for a, c in zip(prev, cur)) / (t_cur - t_prev) / 1e6
                slices.append((rd, wall, t_cur - t_prev))
                cpu_used += cpu_cur - cpu_prev; cpu_wall += t_cur - t_prev
            prev, t_prev, cpu_prev = cur, t_cur, cpu_cur
        if not slices:  # fall back: everything the encoders did so far (or do until they finish, for tiny development clips)
            for p in ps:
                p.wait()
            cur = read()
            rd = sum(c[0] / c[1] for c in cur if c[1] > 0) / 1e6
            slices.append((rd, rd, time.time() - t_start))
    finally:
        for p in ps:  # the encoders we started, by handle
            if p.poll() is None:
                p.kill()
        for p in ps:
            p.wait()
    value = float(np.mean([s[0] for s in slices]))
    res = {"value": round(value, 4), "unit": "Mpixel/s", "cores": nproc, "host_threads": cores, "physical_cores": phys, "kind": "reference",
           "sample": "%d concurrent processes of the unmodified reference encoder (oracle/_ref/Thorenc_capture: SIMD path, gcc -O3 -march=x86-64-v3; the reference "
                     "Makefile uses -march=native) encoding the %dx%d %d-frame clip with %s; measured in %d wall-clock slices of %.1f s after every process finished its I and "
                     "first P frame (%.0f s), from the per-super-block progress the observing shim publishes; value = mean over slices of sum over processes of pixels decided / "
                     "seconds inside the reference's process_block loop%s" % (nproc, cfg.W, cfg.H, nfr, cfg.cfgfile, len(slices), slice_s, settle_s,
                                                                              "; an encoder finished early: whole-run fallback" if early else ""),
           "seconds": round(sum(s[2] for s in slices), 2), "slices_rd_loop_mpixel_s": [round(s[0], 4) for s in slices],
           "wall_clock_value": round(float(np.mean([s[1] for s in slices])), 4),
           "per_thread_mpixel_s": round(value / nproc, 5)}
    # how much CPU the box actually granted: CPU seconds the encoders consumed per wall second of the timed slices; far below `cores` = a shared or quota-limited host
    if not early and cpu_wall > 0:
        eff = cpu_used / cpu_wall
        res["effective_cores"] = round(eff, 1)
        res["mpixel_s_per_effective_core"] = round(value / eff, 4) if eff > 0 else None
    try:
        res["cgroup_cpu_max"] = open("/sys/fs/cgroup/cpu.max").read().strip()
    except Exception:
        pass
    res["note"] = ("value = what this host delivered with one encoder per hardware thread; effective_cores = CPU seconds consumed / wall seconds in the timed slices. "
                   "An unconstrained host scales the one-thread rate (single_stream_reference in the GPU arm's line) by its physical cores at best.")
    try:  # the two arms run back to back on one box: the other arm may reuse this measurement instead of holding the box for minutes again
        json.dump({"time": time.time(), "res": res}, open(os.path.join(tmp, "last_result.json"), "w"))
    except Exception:
        pass
    if brief:
        return res
    line = {"impl": "reference", "metric": cfg.metric(), "value": res["value"], "unit": "Mpixel/s", "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": len(slices),
            "warmup": n_warm, "ms_per_step": round(1e3 * float(np.mean([s[2] for s in slices])), 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8" if cfg.ESZ == 1 else "u16", "data": "synthetic",
            "config": {"workload": cfg.workload(), "frames_per_step": cfg.frames - 1, "parallelism": "%d reference encoder processes on %d host threads" % (nproc, cores),
                       "sample": "one %.1f s slice of the continuously running encoders per step" % slice_s},
            "cpu_baseline": res, "e2e": {"value": res["value"], "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="hdb", choices=sorted(CONFIGS), help="BASELINE.json configuration (default: the headline 1080p HDB_high_efficiency)")
    ap.add_argument("--size", default=None, help="WxH override (development: smaller clips)")
    ap.add_argument("--frames", type=int, default=0, help="clip length override")
    ap.add_argument("--e2e-steps", type=int, default=5, help="steps (GOPs) of the end-to-end launch: min(--steps, this); 0 = --steps")
    ap.add_argument("--cpu-procs", type=int, default=0, help="CPU arm: concurrent reference encoders (0 = one per host thread)")
    ap.add_argument("--cpu-slice", type=float, default=0.0, help="CPU arm: wall-clock seconds per slice (= one step of --impl reference); 0 = 60 s spread over warm-up + steps, "
                                                                  "between 1.5 and 4 s")
    ap.add_argument("--cpu-slices", type=int, default=3, help="CPU arm inside the GPU run (cpu_baseline): timed slices")
    ap.add_argument("--cpu-settle-limit", type=float, default=240.0, help="CPU arm: give up waiting for the steady state after this many seconds")
    ap.add_argument("--cache", default=os.environ.get("THOR_B200_CACHE", "/tmp/thor_b200_bench"))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-fresh", action="store_true", help="cpu_baseline: measure again even if a recent measurement of this box exists in the cache")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the decisions of the last timed step (reconstruction, block state, leaves, coefficients, RD costs) "
                         "as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = Cfg(args.config, tuple(int(v) for v in args.size.split("x")) if args.size else None, args.frames or None)
    os.makedirs(args.cache, exist_ok=True)
    if args.impl == "reference":
        if int(os.environ.get("RANK", 0)) == 0:
            cpu_arm(args, cfg)
        return
    run_gpu(args, cfg)


if __name__ == "__main__":
    main()
