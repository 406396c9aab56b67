// tb_kernels.cuh — __global__ kernels of libthor_b200 (sm_100a).  Block-level kernels: one warp per work item,
// grid-stride over the item array.  Frame-level kernels: one thread per sample / edge, laid out so that lanes walk
// along rows (coalesced 128-byte requests).  See DESIGN.md §4 for the roofline of each kernel.
#pragma once
#include "tb_device.cuh"
#include "../../include/thor_b200.h"

namespace tb {

constexpr int WARPS_PER_CTA = 4;
constexpr int CTA_THREADS = WARPS_PER_CTA * 32;
constexpr int TX_MINBLOCKS = 6;  // __launch_bounds__(128, N) of the transform-chain kernel (measured: 4: 5.84 ms, 5: 5.37, 6: 5.12)
constexpr int ME_MINBLOCKS = 6;  // __launch_bounds__(128, N) of the motion-search kernel: registers/thread <= 65536 / (128 N)

__device__ __forceinline__ int global_warp() { return (blockIdx.x * blockDim.x + threadIdx.x) >> 5; }
__device__ __forceinline__ int total_warps() { return (gridDim.x * blockDim.x) >> 5; }

// ---- a1/a2/a3 --------------------------------------------------------------------------------------------------
// kind 0: SAD, 1: wide SAD (5 x-offsets, first minimum), 2: SSD.  `any_align`: a is not word aligned (unaligned variant)
template <class S>
__global__ void __launch_bounds__(CTA_THREADS) sad_batch_kernel(const tb_sad_item_t *items, int n, int kind, uint32_t *out, int32_t *out2,
                                                                uint64_t *out64) {
  const int lane = lane_id();
  for (int it = global_warp(); it < n; it += total_warps()) {
    tb_sad_item_t q = items[it];
    const S *a = (const S *)q.a, *b = (const S *)q.b;
    if (kind == 2) {
      uint64_t s = warp_ssd<S>(a, q.astride, b, q.bstride, q.width, q.height);
      if (lane == 0) out64[it] = s;
    } else if (kind == 1) {
      const int offs[5] = {-3, -1, 0, 1, 3};
      int roff = lane < 5 ? offs[lane] : 0;
      uint32_t s = multi_sad<S>(a, q.astride, b, q.bstride, q.width, q.height, roff, 5);
      uint32_t best;
      int w = warp_first_min(s, 5, best);
      if (lane == 0) { out[it] = best; out2[it] = offs[w]; }
    } else {
      uint32_t s;
      if ((((uintptr_t)a) & 3) || ((q.astride * (int)sizeof(S)) & 3) || (q.width * (int)sizeof(S)) < 4) {
        // generic path for operands without word alignment
        uint32_t acc = 0;
        const int lw = ilog2(q.width);
        for (int p = lane; p < (q.height << lw); p += 32) {
          int row = p >> lw, col = p & (q.width - 1);
          acc += (uint32_t)iabs((int)a[row * q.astride + col] - (int)b[row * q.bstride + col]);
        }
        s = warp_sum(acc);
      } else
        s = warp_sad<S>(a, q.astride, b, q.bstride, q.width, q.height);
      if (lane == 0) out[it] = s;
    }
  }
}

// a4 single-shot (drop-in shim): which 0 = fasthalf, 1 = fastquarter; res = {sad, x, y}
template <class S>
__global__ void fast_subpel_kernel(const S *a, int as, const S *b, int bs, int w, int h, int which, int fx, int fy, int32_t *res) {
  int bx, by;
  uint32_t s = which ? warp_sad_fastquarter<S>(a, as, b, bs, w, h, fx, fy, bx, by) : warp_sad_fasthalf<S>(a, as, b, bs, w, h, bx, by);
  if (lane_id() == 0) { res[0] = (int32_t)s; res[1] = bx; res[2] = by; }
}

// ---- a5 --------------------------------------------------------------------------------------------------------
// Scheduling of a search batch.  Searches cost ~ area x probes and a batch mixes 4x4 ... 128x128 blocks; a single warp needs
// milliseconds for one 128x128 search.  So blocks of >= 2048 samples are searched by the whole CTA (four warps on four row
// bands, MeTeam), which divides their latency by four: a counting sort (three tiny kernels: histogram, scan, scatter) lists
// them largest first, and one persistent kernel first draws from that list with an atomic cursor (longest-processing-time
// first), then draws the remaining searches, one warp each, from the caller's array in its own order.
// class = ilog2(area), + 16 when the CTA-team form applies (speed 0, height a multiple of 8 rows per warp)
constexpr int ME_TEAM_WARPS = WARPS_PER_CTA;
constexpr int ME_DRAW = 4;
__device__ __forceinline__ int me_class(int w, int h, int speed) {
  const int area = w * h, b = min(ilog2(max(area, 1)), 15);
  return (speed == 0 && area >= 2048 && (h % (8 * ME_TEAM_WARPS)) == 0) ? 16 + b : b;
}
// meta layout (ints): [0,32) histogram, [32,64) first list position of each class, [64,96) fill cursors, 96 = number of team
// items, 97 = team cursor, 98 = warp cursor, 99 = number of listed items, 100 = group cursor.  A class functor returns the
// class (0..31; >= 16: searched/transformed by the whole CTA) of an item, or -1 when the item is not listed.
struct MeClassOf {
  int speed, quad;  // quad: 8-bit samples and speed 0 -> blocks of <= 64 samples are listed too (class 1) and searched four per warp
  __device__ __forceinline__ int operator()(const tb_me_item_t &q) const {
    const int c = me_class(q.width, q.height, speed);
    if (c >= 16) return c;  // team items, largest first
    if (quad && (int)q.width * (int)q.height <= 64 && !((q.width | q.height) & 3) && !(q.ostride & 3) && !(q.rstride & 3) &&
        !((uintptr_t)q.orig & 3))
      return 1;
    return -1;  // the others are drawn from the caller's array in its own order
  }
};
struct TxClassOf {  // transform blocks > 8x8 are listed (one warp each, the CTA for >= 64x64); 4x4 / 8x8 run one per thread
  __device__ __forceinline__ int operator()(const tb_txfm_item_t &q) const { return q.size >= 64 ? 16 + ilog2(q.size) : (q.size > 8 ? ilog2(q.size) : -1); }
};
template <class Item, class F> __global__ void sched_hist_kernel(const Item *items, int n, F f, int *meta) {
  __shared__ int h[32];
  if (threadIdx.x < 32) h[threadIdx.x] = 0;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int c = f(items[i]);
    if (c >= 0) atomicAdd(&h[c], 1);
  }
  __syncthreads();
  if (threadIdx.x < 32 && h[threadIdx.x]) atomicAdd(&meta[threadIdx.x], h[threadIdx.x]);
}
__global__ void sched_scan_kernel(int *meta) {
  const int b = threadIdx.x;  // 32 threads
  int before = 0, team = 0, all = 0;
  for (int k = 31; k > b; k--) before += meta[k];
  for (int k = 0; k < 32; k++) { all += meta[k]; if (k >= 16) team += meta[k]; }
  meta[32 + b] = before;
  meta[64 + b] = 0;
  if (b == 0) { meta[96] = team; meta[97] = 0; meta[98] = 0; meta[99] = all; meta[100] = 0; }
}
template <class Item, class F> __global__ void sched_scatter_kernel(const Item *items, int n, F f, int *meta, int *idx) {
  // warp-aggregated: the lanes of a warp that hold the same class reserve their list positions with ONE atomic
  const int nround = (n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
  for (int k = 0; k < nround; k++) {
    const int i = (k * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
    const int c = i < n ? f(items[i]) : -1;
    const unsigned peers = __match_any_sync(FULL, c);
    int base = 0;
    const int leader = __ffs(peers) - 1;
    if (c >= 0 && lane_id() == leader) base = atomicAdd(&meta[64 + c], __popc(peers));
    base = __shfl_sync(FULL, base, leader);
    if (c >= 0) idx[meta[32 + c] + base + __popc(peers & ((1u << lane_id()) - 1))] = i;
  }
}

template <class S, int TW>
__device__ __noinline__ void me_run_item(const tb_me_item_t *items, int it, const int16_t *cand, int bitdepth, int speed, int bip, int fw, int fh, tb_me_result_t *out,
                                            unsigned long long *stats, MeTeam<TW> &tm) {
  tb_me_item_t q = items[it];
  MeCtx c;
  c.size = q.size; c.width = q.width; c.height = q.height; c.sign = q.sign; c.s = q.sign ? -1 : 1;
  c.xpos = q.xpos; c.ypos = q.ypos; c.fw = fw; c.fh = fh; c.bitdepth = bitdepth; c.speed = speed; c.bip = bip;
  c.mvpx = q.mvp_x; c.mvpy = q.mvp_y; c.lambda = q.lambda; c.n_int = 0; c.n_sub = 0;
  int mx, my;
  uint32_t cost;
  warp_motion_estimate<S, TW>((const S *)q.orig, q.ostride, (const S *)q.ref, q.rstride, c, q.mvc_x, q.mvc_y, cand + 2 * (size_t)q.cand_ofs, q.ncand, mx, my, cost, tm);
  if (lane_id() == 0 && tm.warp == 0) {
    out[it].mvx = (int16_t)mx; out[it].mvy = (int16_t)my; out[it].cost = cost;
    if (stats) {  // roofline accounting (SURVEY.md §8d): samples compared at integer positions, samples fetched for sub-pel probes
      atomicAdd(&stats[0], 1ull);
      atomicAdd(&stats[1], (unsigned long long)c.n_int);
      atomicAdd(&stats[2], (unsigned long long)c.n_sub);
      atomicAdd(&stats[3], (unsigned long long)(c.n_int + 1) * q.width * q.height);
      atomicAdd(&stats[4], (unsigned long long)c.n_sub * ((q.width + 5) * (q.height + 5) + q.width * q.height));
    }
  }
}

template <class S>
__global__ void __launch_bounds__(CTA_THREADS, ME_MINBLOCKS) me_batch_kernel(const tb_me_item_t *items, int n, const int *idx, int *meta, const int16_t *cand, int bitdepth,
                                                                                 int speed, int bip, int fw, int fh, tb_me_result_t *out, unsigned long long *stats) {
  __shared__ uint32_t xch[2 * ME_TEAM_WARPS * 32];
  __shared__ int s_next;
  const int nteam = meta[96], nlisted = meta[99];
  const int quad = sizeof(S) == 1 && speed == 0;
  // phase 1: the CTA as a team on the large blocks
  {
    MeTeam<ME_TEAM_WARPS> tm;
    tm.xch = xch; tm.warp = threadIdx.x >> 5; tm.phase = 0;
    for (;;) {
      if (threadIdx.x == 0) s_next = atomicAdd(&meta[97], 1);
      __syncthreads();
      const int k = s_next;
      __syncthreads();
      if (k >= nteam) break;
      me_run_item<S, ME_TEAM_WARPS>(items, idx[k], cand, bitdepth, speed, bip, fw, fh, out, stats, tm);
    }
  }
  // phase 2: the searches that are neither team nor quad items, one warp each, drawn four at a time from the caller's array
  // (neighbouring items share samples: keep them on neighbouring warps)
  const MeClassOf cls{speed, quad};
  {
    MeTeam<1> tm;
    tm.xch = nullptr; tm.warp = 0; tm.phase = 0;
    for (;;) {
      int k = 0;
      if (lane_id() == 0) k = atomicAdd(&meta[100], ME_DRAW);
      k = __shfl_sync(FULL, k, 0);
      if (k >= n) break;
      for (int it = k; it < min(k + ME_DRAW, n); it++) {
        if (nlisted && cls(items[it]) >= 0) continue;
        me_run_item<S, 1>(items, it, cand, bitdepth, speed, bip, fw, fh, out, stats, tm);
      }
    }
  }
  // phase 3: the listed small blocks (8-bit, <= 64 samples), four per warp (quad_motion_estimate).  They come last: the launch
  // ends on its cheapest searches, and the two code paths do not alternate in the instruction cache.
  if (sizeof(S) == 1) {
    const int nsmall = nlisted - nteam;
    for (;;) {
      int k = 0;
      if (lane_id() == 0) k = atomicAdd(&meta[98], 4);
      k = __shfl_sync(FULL, k, 0);
      if (k >= nsmall) break;
      const int slot = k + (lane_id() >> 3);
      if (slot < nsmall) {
        const int mine = idx[nteam + slot];
        const tb_me_item_t q = items[mine];
        QuadItem qi;
        qi.orig = (const uint8_t *)q.orig; qi.ref = (const uint8_t *)q.ref; qi.cand = cand + 2 * (size_t)q.cand_ofs; qi.lambda = q.lambda;
        qi.os = q.ostride; qi.rs = q.rstride; qi.size = q.size; qi.w = q.width; qi.h = q.height; qi.sign = q.sign; qi.xpos = q.xpos; qi.ypos = q.ypos;
        qi.mvpx = q.mvp_x; qi.mvpy = q.mvp_y; qi.mvcx = q.mvc_x; qi.mvcy = q.mvc_y; qi.ncand = q.ncand;
        int mx, my;
        uint32_t cost;
        unsigned n_int;
        quad_motion_estimate(qi, fw, fh, bip, mx, my, cost, n_int);
        if ((lane_id() & 7) == 0) {
          out[mine].mvx = (int16_t)mx; out[mine].mvy = (int16_t)my; out[mine].cost = cost;
          if (stats) {
            atomicAdd(&stats[0], 1ull);
            atomicAdd(&stats[1], (unsigned long long)n_int);
            atomicAdd(&stats[2], 16ull);
            atomicAdd(&stats[3], (unsigned long long)(n_int + 1) * q.width * q.height);
            atomicAdd(&stats[4], 16ull * ((q.width + 5) * (q.height + 5) + q.width * q.height));
          }
        }
      }
      __syncwarp();
    }
  }
}

template <class S>
__global__ void __launch_bounds__(CTA_THREADS) me_bi_batch_kernel(const tb_me_bi_item_t *items, int n, const int16_t *cand, int bitdepth, int bip, int fw, int fh,
                                                                  tb_me_result_t *out) {
  for (int it = global_warp(); it < n; it += total_warps()) {
    tb_me_bi_item_t q = items[it];
    int mx, my;
    uint32_t cost;
    warp_motion_estimate_bi<S>((const S *)q.orig, q.ostride, (const S *)q.ref0, (const S *)q.ref1, q.rstride, q.size, q.sign, q.xpos, q.ypos, fw, fh, bitdepth, bip, q.lambda,
                               q.mvc_x, q.mvc_y, q.mvp_x, q.mvp_y, cand + 2 * (size_t)q.cand_ofs, q.ncand, mx, my, cost);
    if (lane_id() == 0) { out[it].mvx = (int16_t)mx; out[it].mvy = (int16_t)my; out[it].cost = cost; }
  }
}
// a9 / a5 element-wise block combinations, one warp per item (op 0: (a+b)>>1, 1: sat(2a-b), 2: (a+b+1)>>1)
template <class S> __global__ void __launch_bounds__(CTA_THREADS) combine_batch_kernel(const tb_combine_item_t *items, int n, int op, int bitdepth) {
  const int maxv = (1 << bitdepth) - 1;
  for (int it = global_warp(); it < n; it += total_warps()) {
    tb_combine_item_t q = items[it];
    const S *a = (const S *)q.a, *b = (const S *)q.b;
    S *d = (S *)q.dst;
    for (int p = lane_id(); p < q.width * q.height; p += 32) {
      int row = p / q.width, col = p - row * q.width;
      int x = a[row * q.astride + col], y = b[row * q.bstride + col];
      int v = op == 0 ? (x + y) >> 1 : (op == 1 ? sat_px(2 * x - y, maxv) : (x + y + 1) >> 1);
      d[row * q.dstride + col] = (S)v;
    }
  }
}

// ---- a7/a8 -----------------------------------------------------------------------------------------------------
// Four consecutive items per warp and step.  85 % of the predictions of an encode are blocks of <= 64 samples (4x4 ... 8x8 luma,
// 2x2 ... 8x8 chroma) whose cost is one dependent chain item -> samples -> store: when all four are that small, each gets a group
// of eight lanes and the four chains overlap; otherwise the warp takes them one after the other.  (Eight groups of four lanes for
// blocks of <= 16 samples were measured slower: 96 registers instead of 72, 1.81 ms instead of 1.57 ms for the 1080p batch.)
template <class S> __global__ void __launch_bounds__(CTA_THREADS) interp_batch_kernel(const tb_interp_item_t *items, int n, int bitdepth, int bip) {
  const int lane = lane_id(), grp = lane >> 3;
  for (int base = global_warp() * 4; base < n; base += total_warps() * 4) {
    const int mine = base + grp;
    tb_interp_item_t q;
    bool small = true;
    if (mine < n) {
      q = items[mine];
      small = (int)q.width * (int)q.height <= 64;
    }
    if (__all_sync(FULL, small)) {
      if (mine < n)
        warp_interp<S>((S *)q.dst, q.dstride, (const S *)q.ref, q.rstride, q.width, q.height, q.mvx, q.mvy, q.sign, q.chroma, q.chroma ? 0 : bip, q.pic_w, q.pic_h, q.xpos,
                       q.ypos, bitdepth, lane & 7, 8);
    } else {
      for (int it = base; it < min(base + 4, n); it++) {
        const tb_interp_item_t t = items[it];
        warp_interp<S>((S *)t.dst, t.dstride, (const S *)t.ref, t.rstride, t.width, t.height, t.mvx, t.mvy, t.sign, t.chroma, t.chroma ? 0 : bip, t.pic_w, t.pic_h, t.xpos,
                       t.ypos, bitdepth);
      }
    }
    __syncwarp();
  }
}
// fractional-offset form of the drop-in symbols (ip already at the integer position)
template <class S>
__global__ void interp_frac_kernel(S *dst, int ds, const S *ip, int is, int w, int h, int xf, int yf, int chroma, int bip, int bitdepth) {
  const int maxv = (1 << bitdepth) - 1, lw = ilog2(w);
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < (h << lw); p += gridDim.x * blockDim.x) {
    int row = p >> lw, col = p & (w - 1);
    const S *q = ip + row * is + col;
    dst[row * ds + col] = (S)(chroma ? chroma_sample<S>(q, is, xf, yf, maxv) : luma_sample<S>(q, is, xf, yf, bip, maxv));
  }
}
template <class S> __global__ void block_avg_kernel(S *p, int sp, const S *r0, int s0, const S *r1, int s1, int w, int h) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x) {
    int row = i / w, col = i % w;
    p[row * sp + col] = (S)up2(r0[row * s0 + col], r1[row * s1 + col]);
  }
}

// ---- a10-a13 + a3 ----------------------------------------------------------------------------------------------
struct alignas(16) TxShared {
  TxScratch sc;
};

constexpr int TX_TABLE_BYTES = (DCT_TAB8_SIZE * 2 + 256 + 15) & ~15;  // int8 matrices (plain, transposed) + 16x16 zig-zag table
// residual on the fly -> forward -> quantise -> de-quantise -> inverse -> reconstruct + SSD.
// One transform block > 8x8 handled by a team of TW warps (TW == 1: a warp; TW == WARPS_PER_CTA: the CTA, for 64x64 and
// 128x128 whose box-sum load and replicated output are per-sample passes over up to 16384 samples).
template <class S, int TW>
__device__ __noinline__ void tx_big_chain(const tb_txfm_item_t &q, int bitdepth, TxScratch &sc, int16_t *rt, const int8_t *tab8, const int8_t *tab8t, unsigned long long *red,
                                          int *bc, tb_txfm_result_t *res) {
  const uint8_t *zz16 = (const uint8_t *)(tab8 + 2 * DCT_TAB8_SIZE);  // 16x16 zig-zag table behind the two matrix tables
  constexpr int PI = 40;  // int16 pitch of the scratch tiles: 80-byte rows (16-byte aligned; eight consecutive rows cover all 32 banks with 128-bit loads)
  constexpr int NT = 32 * TW;
  const int tid = TW == 1 ? lane_id() : (int)threadIdx.x, lane = lane_id(), maxv = (1 << bitdepth) - 1;
  auto sync = [&]() { if (TW == 1) __syncwarp(); else __syncthreads(); };
  const S *orig = (const S *)q.orig, *pred = (const S *)q.pred;
  S *rec = (S *)q.rec;
  const int size = q.size;
  int size1 = size, scale = 1;
  const int fast = q.fast & 1, want_bits = q.fast & 2;  // flags byte: TB_TXFM_FAST | TB_TXFM_BITS
  if (size > (32 >> fast)) { size1 = 32 >> fast; scale = size / size1; }
  const int l1 = ilog2(size1), qsize = min(size, 16), lq = ilog2(qsize);
  const int8_t *M1 = tab8 + dct_tab8_ofs(l1);
  const int mp1 = dct_tab8_pitch(l1);
  // residual (enc/encode_block.c:162-171) fused with the box-sum load of the forward transform (common/transform.c:261-278:
  // the sum saturates after every addition, rows outer / columns inner)
  if (scale == 1) {
    for (int p = tid; p < (size1 * size1) >> 2; p += NT) {  // four samples per thread and step
      int i = p >> (l1 - 2), j = (p & ((size1 >> 2) - 1)) << 2;
      int a[4], b[4];
      load_row4<S>(orig + i * q.ostride + j, a);
      load_row4<S>(pred + i * q.pstride + j, b);
      *(uint2 *)&sc.in[i * PI + j] = make_uint2(((uint32_t)(a[0] - b[0]) & 0xffffu) | ((uint32_t)(a[1] - b[1]) << 16), ((uint32_t)(a[2] - b[2]) & 0xffffu) | ((uint32_t)(a[3] - b[3]) << 16));
    }
  } else if (scale == 4) {
    for (int p = tid; p < size1 * size1; p += NT) {
      int i = p >> l1, j = p & (size1 - 1), sum = 0;
      for (int m = 0; m < 4; m++) {
        int a[4], b[4];
        load_row4<S>(orig + (i * 4 + m) * q.ostride + j * 4, a);
        load_row4<S>(pred + (i * 4 + m) * q.pstride + j * 4, b);
#pragma unroll
        for (int t = 0; t < 4; t++) sum = iclip(sum + (a[t] - b[t]), -16384, 16383);
      }
      sc.in[i * PI + j] = (int16_t)sum;
    }
  } else if (scale == 2) {
    for (int p = tid; p < (size1 * size1) >> 1; p += NT) {  // two outputs (four source columns) per thread and step
      int i = p >> (l1 - 1), j = (p & ((size1 >> 1) - 1)) << 1, s0 = 0, s1 = 0;
      for (int m = 0; m < 2; m++) {
        int a[4], b[4];
        load_row4<S>(orig + (i * 2 + m) * q.ostride + j * 2, a);
        load_row4<S>(pred + (i * 2 + m) * q.pstride + j * 2, b);
        s0 = iclip(s0 + (a[0] - b[0]), -16384, 16383); s0 = iclip(s0 + (a[1] - b[1]), -16384, 16383);
        s1 = iclip(s1 + (a[2] - b[2]), -16384, 16383); s1 = iclip(s1 + (a[3] - b[3]), -16384, 16383);
      }
      sc.in[i * PI + j] = (int16_t)s0;
      sc.in[i * PI + j + 1] = (int16_t)s1;
    }
  } else {
    for (int p = tid; p < size1 * size1; p += NT) {
      int i = p >> l1, j = p & (size1 - 1), sum = 0;
      for (int m = 0; m < scale; m++)
        for (int nn = 0; nn < scale; nn++) {
          int y = i * scale + m, x = j * scale + nn;
          sum = iclip(sum + ((int)orig[y * q.ostride + x] - (int)pred[y * q.pstride + x]), -16384, 16383);
        }
      sc.in[i * PI + j] = (int16_t)sum;
    }
  }
  sync();
  // The transform phases run on one warp (the first warp of a team: they are a small part of a 64x64/128x128 chain).  Lane
  // (ia = lane >> 3, jb = lane & 7) owns the outputs {4 ia .. 4 ia + 3} x {jb, jb + 8, ..}: the matrix rows are uniform per
  // quarter-warp (broadcast) and the vectors of a quarter-warp are eight consecutive 80-byte rows (conflict-free).
  const bool dct_warp = TW == 1 || threadIdx.x < 32;
  const int ia = lane >> 3, jb = lane & 7;
  {
    const int shift1 = ilog2(size) + ilog2(scale) + bitdepth - 8, add1 = 1 << (shift1 - 1);
    const int shift2 = l1 + 5, add2 = 1 << (shift2 - 1);
    // tmp[i][j] = (M[i][.] . in[j][.] + add1) >> shift1   (i < 16, j < size1)
    if (dct_warp) {
      if (size1 == 16) {
        int acc[4][2] = {};
        dot16_block<4, 2>(M1 + 4 * ia * mp1, mp1, sc.in + jb * PI, 8 * PI, acc);
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
          for (int c = 0; c < 2; c++) sc.tmp[(4 * ia + r) * PI + jb + 8 * c] = (int16_t)((acc[r][c] + add1) >> shift1);
      } else {
        int acc[4][4] = {};
        dot16_block<4, 4>(M1 + 4 * ia * mp1, mp1, sc.in + jb * PI, 8 * PI, acc);
        dot16_block<4, 4>(M1 + 4 * ia * mp1 + 16, mp1, sc.in + jb * PI + 16, 8 * PI, acc);
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
          for (int c = 0; c < 4; c++) sc.tmp[(4 * ia + r) * PI + jb + 8 * c] = (int16_t)((acc[r][c] + add1) >> shift1);
      }
    }
    sync();
    // coef[i][j] = (M[i][.] . tmp[j][.] + add2) >> shift2  (i, j < 16)
    if (dct_warp) {
      int acc[4][2] = {};
      dot16_block<4, 2>(M1 + 4 * ia * mp1, mp1, sc.tmp + jb * PI, 8 * PI, acc);
      if (size1 == 32) dot16_block<4, 2>(M1 + 4 * ia * mp1 + 16, mp1, sc.tmp + jb * PI + 16, 8 * PI, acc);
#pragma unroll
      for (int r = 0; r < 4; r++)
#pragma unroll
        for (int c = 0; c < 2; c++) sc.rc[(4 * ia + r) * 16 + jb + 8 * c] = (int16_t)((acc[r][c] + add2) >> shift2);
    }
    sync();
  }
  int cbp;
  if (TW == 1) cbp = warp_quantize(sc.rc, sc.cq, q.qp, size, q.coeff_type, sc, zz16);
  else {
    if (threadIdx.x < 32) {
      int c = warp_quantize(sc.rc, sc.cq, q.qp, size, q.coeff_type, sc, zz16);
      if (lane == 0) *bc = c;
    }
    __syncthreads();
    cbp = *bc;
  }
  if (q.coeffq)
    for (int p = tid; p < qsize * qsize; p += NT) q.coeffq[p] = sc.cq[p];
  int bits = 0;
  if (want_bits && cbp && dct_warp) bits = warp_coeff_bits(sc.tmp, qsize * qsize, size, q.coeff_type);  // sc.tmp: the levels in scan order (warp_quantize)
  uint64_t ssd = 0;
  if (cbp) {
    // de-quantise (common/common_block.c:45-73) straight into the TRANSPOSED tile in[i][k] = rcoeff[k][i], so that the
    // inverse transform's sums over k read contiguous int16 pairs
    {
      const int lshift = q.qp / 6, rshift = ilog2(size) - 1;
      const int dscale = c_dequant[q.qp % 6];  // |c * dscale| <= 32768 * 72 and the shift is <= qp / 6: 32-bit arithmetic is exact
      const int dadd = lshift < rshift ? (1 << (rshift - lshift - 1)) : 0;
      for (int p = tid; p < qsize * qsize; p += NT) {
        int k = p >> lq, i = p & (qsize - 1), c = sc.cq[p];
        sc.in[i * PI + k] = lshift >= rshift ? (int16_t)((unsigned)(c * dscale) << (lshift - rshift)) : (int16_t)((c * dscale + dadd) >> (rshift - lshift));
      }
      sync();
    }
    // inverse transform with the reconstruction (common/common_block.c:75-83) and SSD fused into its output stage
    const int core = min(size, 32), rep = size / core, lc = ilog2(core);
    const int shiftB = 20 - bitdepth, addB = 1 << (shiftB - 1);
    const int8_t *Mt = tab8t + dct_tab8_ofs(lc);
    const int mpc = dct_tab8_pitch(lc);
    // T[i][j] = clip16((sum_k M[k][j] * rcoeff[k][i] + 64) >> 7), stored transposed: tmp2[j][i]   (i < 16, j < core)
    int16_t *tmp2 = sc.in + 16 * PI;  // rows 16.. of the `in` tile are free here (rcoeff^T uses rows 0..15)
    if (dct_warp) {
      if (core == 16) {
        int acc[4][2] = {};
        dot16_block<4, 2>(Mt + 4 * ia * mpc, mpc, sc.in + jb * PI, 8 * PI, acc);
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
          for (int c = 0; c < 2; c++) tmp2[(4 * ia + r) * PI + jb + 8 * c] = (int16_t)iclip((acc[r][c] + 64) >> 7, -32768, 32767);
      } else {
#pragma unroll
        for (int half = 0; half < 2; half++) {
          int acc[4][2] = {};
          dot16_block<4, 2>(Mt + (16 * half + 4 * ia) * mpc, mpc, sc.in + jb * PI, 8 * PI, acc);
#pragma unroll
          for (int r = 0; r < 4; r++)
#pragma unroll
            for (int c = 0; c < 2; c++) tmp2[(16 * half + 4 * ia + r) * PI + jb + 8 * c] = (int16_t)iclip((acc[r][c] + 64) >> 7, -32768, 32767);
        }
      }
    }
    sync();
    // out[i][j] = clip16((sum_k M[k][j] * T[k][i] + addB) >> shiftB) = Mt[j][.] . tmp2[i][.]   (i, j < core); lane (jg = lane >> 3,
    // il = lane & 7) owns columns 4 jg .. 4 jg + 3 (+16 in a second pass for core 32) of rows il, il + 8, ..
    if (rep == 1) {
      if (dct_warp) {
        for (int jg = ia; jg < (core >> 2); jg += 4) {
          for (int i0 = jb; i0 < core; i0 += 16) {
            int acc[4][2] = {};
            dot16_block<4, 2>(Mt + 4 * jg * mpc, mpc, tmp2 + i0 * PI, 8 * PI, acc);
#pragma unroll
            for (int c = 0; c < 2; c++) {
              const int i = i0 + 8 * c, j = 4 * jg;
              int pv[4], ov[4], v[4];
              load_row4<S>(pred + i * q.pstride + j, pv);
              load_row4<S>(orig + i * q.ostride + j, ov);
#pragma unroll
              for (int t = 0; t < 4; t++) {
                int r = iclip((acc[t][c] + addB) >> shiftB, -32768, 32767);
                v[t] = sat_px(r + pv[t], maxv);
                int d = ov[t] - v[t];
                ssd += (uint64_t)(uint32_t)(d * d);
              }
              if (rec) store_row4<S>(rec + i * q.rstride + j, v);
            }
          }
        }
      }
    } else if (TW > 1 && (rep == 2 || rep == 4)) {
      // the core x core residual goes to a second tile, then one per-sample pass replicates it (common/transform.c:481-492)
      if (dct_warp) {
        for (int jg = ia; jg < (core >> 2); jg += 4) {
          for (int i0 = jb; i0 < core; i0 += 16) {
            int acc[4][2] = {};
            dot16_block<4, 2>(Mt + 4 * jg * mpc, mpc, tmp2 + i0 * PI, 8 * PI, acc);
#pragma unroll
            for (int c = 0; c < 2; c++)
#pragma unroll
              for (int t = 0; t < 4; t++) rt[(i0 + 8 * c) * PI + 4 * jg + t] = (int16_t)iclip((acc[t][c] + addB) >> shiftB, -32768, 32767);
          }
        }
      }
      __syncthreads();
      const int ls = ilog2(size), lr = ilog2(rep);
      for (int p = tid; p < (size * size) >> 2; p += NT) {
        int y = p >> (ls - 2), x = (p & ((size >> 2) - 1)) << 2;
        int pv[4], ov[4], v[4];
        load_row4<S>(pred + y * q.pstride + x, pv);
        load_row4<S>(orig + y * q.ostride + x, ov);
        const int16_t *rr = rt + (y >> lr) * PI;
#pragma unroll
        for (int t = 0; t < 4; t++) {
          v[t] = sat_px((int)rr[(x + t) >> lr] + pv[t], maxv);
          int d = ov[t] - v[t];
          ssd += (uint64_t)(uint32_t)(d * d);
        }
        if (rec) store_row4<S>(rec + y * q.rstride + x, v);
      }
    } else {
      for (int p = tid; p < core * core; p += NT) {
        int i = p >> lc, j = p & (core - 1);
        int sum = dot_s8_s16(Mt + j * mpc, tmp2 + i * PI, qsize);
        int r = iclip((sum + addB) >> shiftB, -32768, 32767);
        for (int m = 0; m < rep; m++)
          for (int nn = 0; nn < rep; nn++) {
            int y = i * rep + m, x = j * rep + nn;
            int v = sat_px(r + (int)(int16_t)pred[y * q.pstride + x], maxv);
            if (rec) rec[y * q.rstride + x] = (S)v;
            int d = (int)orig[y * q.ostride + x] - v;
            ssd += (uint64_t)(uint32_t)(d * d);
          }
      }
    }
  } else {
    // cbp == 0: the reference copies the prediction (enc/encode_block.c:1145-1166 "memcpy pred -> rec")
    const int ls = ilog2(size);
    for (int p = tid; p < (size * size) >> 2; p += NT) {
      int y = p >> (ls - 2), x = (p & ((size >> 2) - 1)) << 2;
      int pv[4], ov[4];
      load_row4<S>(pred + y * q.pstride + x, pv);
      load_row4<S>(orig + y * q.ostride + x, ov);
      if (rec) store_row4<S>(rec + y * q.rstride + x, pv);
#pragma unroll
      for (int t = 0; t < 4; t++) { int d = ov[t] - pv[t]; ssd += (uint64_t)(uint32_t)(d * d); }
    }
  }
  ssd = warp_sum64(ssd);
  if (TW > 1) {
    if (lane == 0) red[threadIdx.x >> 5] = ssd;
    __syncthreads();
    ssd = 0;
#pragma unroll
    for (int k = 0; k < TW; k++) ssd += red[k];
  }
  if (tid == 0) { res->ssd = ssd; res->cbp = cbp; res->bits = bits; }
  sync();
}

// Scheduling as for the motion search (me_batch_kernel): blocks > 8x8 are listed largest first by the counting sort; the
// persistent kernel (1) works through the 64x64 / 128x128 blocks as a CTA team, (2) gives the 16x16 / 32x32 blocks one warp
// each, (3) draws groups of 32 consecutive items from the caller's array and runs their 4x4 and 8x8 blocks one per LANE
// (thread_txfm4 in registers, thread_txfm8 in per-thread local arrays; consecutive items are spatial neighbours, so the
// lanes' loads and stores coalesce).
template <class S>
__global__ void __launch_bounds__(CTA_THREADS, TX_MINBLOCKS) txfm_chain_kernel(const tb_txfm_item_t *items, int n, const int *idx, int *meta, int bitdepth, tb_txfm_result_t *out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned long long red[WARPS_PER_CTA];
  __shared__ int bc, s_next;
  int8_t *tab8 = (int8_t *)smem_raw, *tab8t = tab8 + DCT_TAB8_SIZE;
  TxScratch *scs = (TxScratch *)(smem_raw + TX_TABLE_BYTES);
  dct_tab8_fill(tab8, tab8t);
  for (int t = threadIdx.x; t < 256; t += blockDim.x) ((uint8_t *)(tab8 + 2 * DCT_TAB8_SIZE))[t] = (uint8_t)zigzag_index(t >> 4, t & 15, 16);
  __syncthreads();
  const int lane = lane_id();
  const int nteam = meta[96], nlisted = meta[99];
  for (;;) {  // (1)
    if (threadIdx.x == 0) s_next = atomicAdd(&meta[97], 1);
    __syncthreads();
    const int k = s_next;
    __syncthreads();
    if (k >= nteam) break;
    const int it = idx[k];
    tx_big_chain<S, WARPS_PER_CTA>(items[it], bitdepth, scs[0], scs[1].in, tab8, tab8t, red, &bc, out + it);
  }
  TxScratch &sc = scs[threadIdx.x >> 5];
  for (;;) {  // (2)
    int k = 0;
    if (lane == 0) k = atomicAdd(&meta[98], 1);
    k = nteam + __shfl_sync(FULL, k, 0);
    if (k >= nlisted) break;
    const int it = idx[k];
    tx_big_chain<S, 1>(items[it], bitdepth, sc, nullptr, tab8, tab8t, nullptr, nullptr, out + it);
  }
  const int ngroups = (n + 31) >> 5;
  for (;;) {  // (3)
    int gidx = 0;
    if (lane == 0) gidx = atomicAdd(&meta[100], 1);
    gidx = __shfl_sync(FULL, gidx, 0);
    if (gidx >= ngroups) break;
    const int mine = gidx * 32 + lane;
    int my_size = 0;
    if (mine < n) my_size = items[mine].size;
    if (my_size == 4) {
      tb_txfm_item_t q = items[mine];
      uint64_t ssd;
      int bits;
      int cbp = thread_txfm4<S>((const S *)q.orig, q.ostride, (const S *)q.pred, q.pstride, (S *)q.rec, q.rstride, q.coeffq, q.qp, q.coeff_type, bitdepth, ssd, q.fast & 2, bits);
      out[mine].ssd = ssd; out[mine].cbp = cbp; out[mine].bits = bits;
    } else if (my_size == 8) {
      tb_txfm_item_t q = items[mine];
      uint64_t ssd;
      int bits;
      int cbp = thread_txfm8<S>((const S *)q.orig, q.ostride, (const S *)q.pred, q.pstride, (S *)q.rec, q.rstride, q.coeffq, q.qp, q.coeff_type, bitdepth, tab8, tab8t, ssd,
                                q.fast & 2, bits);
      out[mine].ssd = ssd; out[mine].cbp = cbp; out[mine].bits = bits;
    }
    __syncwarp();
  }
}

// drop-in single-shot kernels (one warp)
__global__ void fwd_transform_kernel(const int16_t *block, int16_t *coeff, int size, int fast, int bitdepth) {
  __shared__ TxShared sh;
  __shared__ int16_t tab[DCT_TAB_SIZE];
  dct_tab_fill(tab);
  __syncthreads();
  const int qsize = min(size, 16);
  warp_fwd_transform(block, size, size, fast, bitdepth, sh.sc, sh.sc.rc, tab);
  for (int p = lane_id(); p < qsize * qsize; p += 32) coeff[(p / qsize) * size + (p % qsize)] = sh.sc.rc[p];
}
__global__ void inv_transform_kernel(const int16_t *coeff, int16_t *block, int size, int bitdepth) {
  __shared__ TxShared sh;
  __shared__ int16_t tab[DCT_TAB_SIZE];
  dct_tab_fill(tab);
  __syncthreads();
  const int qsize = min(size, 16);
  for (int p = lane_id(); p < qsize * qsize; p += 32) sh.sc.rc[p] = coeff[(p / qsize) * size + (p % qsize)];
  __syncwarp();
  warp_inv_transform(sh.sc.rc, qsize, size, bitdepth, sh.sc, block, size, tab);
}
__global__ void quant_kernel(const int16_t *coeff, int16_t *coeffq, int qp, int size, int type, int32_t *cbp) {
  __shared__ TxShared sh;
  const int qsize = min(size, 16);
  for (int p = lane_id(); p < qsize * qsize; p += 32) sh.sc.rc[p] = coeff[(p / qsize) * size + (p % qsize)];
  __syncwarp();
  int c = warp_quantize(sh.sc.rc, sh.sc.cq, qp, size, type, sh.sc);
  for (int p = lane_id(); p < qsize * qsize; p += 32) coeffq[p] = sh.sc.cq[p];
  if (lane_id() == 0) *cbp = c;
}
__global__ void dequant_kernel(const int16_t *coeffq, int16_t *rcoeff, int qp, int size) {
  __shared__ TxShared sh;
  const int qsize = min(size, 16);
  warp_dequantize(coeffq, sh.sc.rc, qp, size);
  for (int p = lane_id(); p < qsize * qsize; p += 32) rcoeff[(p / qsize) * size + (p % qsize)] = sh.sc.rc[p];
}
__global__ void calc_cbp_kernel(const int16_t *block, int size, int thr, int32_t *res) {
  int r = warp_calc_cbp(block, size, thr);
  if (lane_id() == 0) *res = r;
}
__global__ void check_nz_kernel(const int16_t *coeff, int size, int32_t *res) {
  int r = warp_check_nz_area(coeff, size);
  if (lane_id() == 0) *res = r;
}

// ---- a15/a16 ---------------------------------------------------------------------------------------------------
template <class S> struct IntraShared {
  S left[256], top[256], filt[4 * 128 + 4];
};
template <class S> __global__ void __launch_bounds__(CTA_THREADS) intra_batch_kernel(const tb_intra_item_t *items, int n, int bitdepth) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  IntraShared<S> &sh = ((IntraShared<S> *)smem_raw)[threadIdx.x >> 5];
  for (int it = global_warp(); it < n; it += total_warps()) {
    tb_intra_item_t q = items[it];
    S tl;
    warp_make_top_and_left<S>(sh.left, sh.top, tl, (const S *)q.rec, q.rstride, (const S *)nullptr, 0, 0, 0, q.ypos, q.xpos, q.size, q.upright, q.downleft, 0,
                              bitdepth);
    warp_intra_pred<S>(sh.left, sh.top, tl, q.ypos, q.xpos, q.size, (S *)q.dst, q.size, q.mode, bitdepth, sh.filt);
  }
}
template <class S> __global__ void cfl_kernel(const S *y, S *u, S *v, const S *ry, int n, int cstride, int stride, int sub, int bitdepth) {
  warp_cfl<S>(y, u, v, ry, n, cstride, stride, sub, bitdepth);
}

// ---- a17: deblocking ------------------------------------------------------------------------------------------
__constant__ uint8_t c_beta[52] = {0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15,
                                   16, 17, 18, 20, 22, 24, 26, 28, 30, 32, 34, 36, 38, 40, 42, 44, 46, 48, 50, 52, 54, 56, 58, 60, 62, 64};
__constant__ uint8_t c_tc[56] = {0,  0,  1,  1,  2,  3,  4,  5,  6,  7,  8,  9,  10,  11,  12,  13,  14,  15,  16,
                                 17, 18, 20, 22, 24, 26, 28, 30, 32, 36, 40, 44, 48,  52,  56,  60,  64,  68,  72,
                                 80, 88, 96, 104, 112, 128, 144, 152, 160, 168, 176, 184, 192, 200, 208, 216, 224, 232};

__device__ __forceinline__ bool db_edge_on(const tb_blkinfo_t &q, const tb_blkinfo_t &p, int pos, int vertical) {
  int q_size = q.size;
  bool part_hit = vertical ? (q.pb_part == 2 || q.pb_part == 3) : (q.pb_part == 1 || q.pb_part == 3);
  if ((q.tb_split || part_hit) && q_size > 8) q_size >>= 1;
  bool mv = iabs(p.mv0y) >= 4 || iabs(q.mv0y) >= 4 || iabs(p.mv0x) >= 4 || iabs(q.mv0x) >= 4 || iabs(p.mv1y) >= 4 || iabs(q.mv1y) >= 4 ||
            iabs(p.mv1x) >= 4 || iabs(q.mv1x) >= 4;
  bool cbp = p.cbp_y || q.cbp_y, intra = p.mode == 1 || q.mode == 1;
  bool interior = q_size ? (pos % q_size) > 0 : false;
  return !interior && (mv || cbp || intra);
}

// Vertical edges (common/common_frame.c:84-200): one thread per 8-row edge segment; lanes walk along x so the 32
// edges of a warp touch one 256-byte span per row.
template <class S>
__global__ void deblock_y_vert_kernel(S *rec, int stride, const tb_blkinfo_t *bi, int width, int height, int beta, int tc, int maxv) {
  const int ex = blockIdx.x * blockDim.x + threadIdx.x;  // edge index along x: j = 8 * (ex + 1)
  const int i = (blockIdx.y * blockDim.y + threadIdx.y) * 8;
  const int j = 8 * (ex + 1);
  if (j >= width || i >= height) return;
  S *p = rec + i * stride + j;
  int px[8][4];
#pragma unroll
  for (int k = 0; k < 8; k++)
#pragma unroll
    for (int t = 0; t < 4; t++) px[k][t] = p[k * stride + t - 2];
  auto act = [&](int k) { return iabs(px[k][0] - px[k][1]) + iabs(px[k][3] - px[k][2]); };
  const int d15 = act(1) + act(5), d26 = act(2) + act(6);
  const int bw = width >> 2;
#pragma unroll
  for (int m = 0; m < 8; m += 4) {
    const tb_blkinfo_t q = bi[((i + m) >> 2) * bw + (j >> 2)], pp = bi[((i + m) >> 2) * bw + (j >> 2) - 1];
    if (!db_edge_on(q, pp, j, 1)) continue;
#pragma unroll
    for (int k = m; k < m + 4; k++) {
      int d = (k & 1) ? d26 : d15;
      if (d >= beta) continue;
      int p1 = px[k][0], p0 = px[k][1], q0 = px[k][2], q1 = px[k][3];
      int delta = iclip((18 * (q0 - p0) - 6 * (q1 - p1) + 16) >> 5, -tc, tc);
      p[k * stride - 2] = (S)sat_px(p1 + delta / 2, maxv);
      p[k * stride - 1] = (S)sat_px(p0 + delta, maxv);
      p[k * stride + 0] = (S)sat_px(q0 - delta, maxv);
      p[k * stride + 1] = (S)sat_px(q1 - delta / 2, maxv);
    }
  }
}
// Horizontal edges (:203-351): one thread per column; the 8 lanes of an edge share the two activity sums.
template <class S>
__global__ void deblock_y_horz_kernel(S *rec, int stride, const tb_blkinfo_t *bi, int width, int height, int beta, int tc, int maxv) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = 8 * (blockIdx.y + 1);
  if (i >= height) return;
  const bool live = x < width;
  S *p = rec + i * stride + (live ? x : 0);
  int p1 = p[-2 * stride], p0 = p[-stride], q0 = p[0], q1 = p[stride];
  int a = iabs(p1 - p0) + iabs(q1 - q0);
  const int l8 = lane_id() & ~7;
  int d15 = __shfl_sync(FULL, a, l8 + 1) + __shfl_sync(FULL, a, l8 + 5);
  int d26 = __shfl_sync(FULL, a, l8 + 2) + __shfl_sync(FULL, a, l8 + 6);
  if (!live) return;
  const int bw = width >> 2;
  const tb_blkinfo_t q = bi[(i >> 2) * bw + (x >> 2)], pp = bi[((i >> 2) - 1) * bw + (x >> 2)];
  if (!db_edge_on(q, pp, i, 0)) return;
  int d = (x & 1) ? d26 : d15;
  if (d >= beta) return;
  int delta = iclip((18 * (q0 - p0) - 6 * (q1 - p1) + 16) >> 5, -tc, tc);
  p[-2 * stride] = (S)sat_px(p1 + delta / 2, maxv);
  p[-stride] = (S)sat_px(p0 + delta, maxv);
  p[0] = (S)sat_px(q0 - delta, maxv);
  p[stride] = (S)sat_px(q1 - delta / 2, maxv);
}
// Chroma (common/common_frame.c:354-432): pass 0 vertical edges, pass 1 horizontal; one thread per chroma sample
// along the edge.  width/height are luma dimensions.
template <class S>
__global__ void deblock_uv_kernel(S *recU, S *recV, int stride, const tb_blkinfo_t *bi, int width, int height, int pass, int tc, int maxv) {
  S *c = blockIdx.z ? recV : recU;
  const int bw = width >> 2;
  if (pass == 0) {
    const int y2 = blockIdx.y * blockDim.y + threadIdx.y;            // chroma row
    const int j = 8 * (blockIdx.x * blockDim.x + threadIdx.x + 1);   // luma edge column
    if (j >= width || y2 >= (height >> 1)) return;
    const int i = (y2 >> 2) << 3;
    const tb_blkinfo_t q = bi[(i >> 2) * bw + (j >> 2)], p = bi[(i >> 2) * bw + (j >> 2) - 1];
    if (!((p.mode == 1 || q.mode == 1) && (q.size ? (j % q.size) == 0 : true))) return;
    S *s = c + y2 * stride + (j >> 1);
    int p1 = s[-2], p0 = s[-1], q0 = s[0], q1 = s[1];
    int delta = iclip((4 * (q0 - p0) + (p1 - q1) + 4) >> 3, -tc, tc);
    s[-1] = (S)sat_px(p0 + delta, maxv);
    s[0] = (S)sat_px(q0 - delta, maxv);
  } else {
    const int x2 = blockIdx.x * blockDim.x + threadIdx.x;  // chroma column
    const int i = 8 * (blockIdx.y + 1);
    if (i >= height || x2 >= (width >> 1)) return;
    const int j = (x2 >> 2) << 3;
    const tb_blkinfo_t q = bi[(i >> 2) * bw + (j >> 2)], p = bi[((i >> 2) - 1) * bw + (j >> 2)];
    if (!((p.mode == 1 || q.mode == 1) && (q.size ? (i % q.size) == 0 : true))) return;
    S *s = c + (i >> 1) * stride + x2;
    int p1 = s[-2 * stride], p0 = s[-stride], q0 = s[0], q1 = s[stride];
    int delta = iclip((4 * (q0 - p0) + (p1 - q1) + 4) >> 3, -tc, tc);
    s[-stride] = (S)sat_px(p0 + delta, maxv);
    s[0] = (S)sat_px(q0 - delta, maxv);
  }
}

// ---- a18: CLPF -------------------------------------------------------------------------------------------------
// per filter block "all skip" flags with the reference's index arithmetic (common/common_frame.c:1042-1053):
// grid pitch = plane width / 4 (sic).  width,height = plane dimensions.
__global__ void clpf_allskip_kernel(const tb_blkinfo_t *bi, int width, int height, int sub, int fb_size_log2, uint8_t *allskip) {
  const int bs = sub ? 4 : 8, fb = 1 << fb_size_log2;
  const int nh = (width + fb - 1) >> fb_size_log2, nv = (height + fb - 1) >> fb_size_log2;
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nh * nv) return;
  const int xoff = (f % nh) << fb_size_log2, yoff = (f / nh) << fb_size_log2;
  int all = 1;
  for (int m = 0; all && m < fb / bs; m++)
    for (int n = 0; all && n < fb / bs; n++) {
      int xpos = xoff + n * bs, ypos = yoff + m * bs;
      if (xpos < width && ypos < height) all &= bi[((ypos << sub) / 4) * (width / 4) + ((xpos << sub) / 4)].mode == 0;
    }
  allskip[f] = (uint8_t)all;
}
// out-of-place plane filter: every read sees unfiltered samples (DESIGN.md §3.4).  One thread per sample.
template <class S>
__global__ void clpf_plane_kernel(const S *src, S *dst, int stride, int width, int height, const tb_blkinfo_t *bi, int sub, const uint8_t *allskip,
                                  const uint8_t *fb_on, int fb_size_log2, int strength, int damping) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= width || y >= height) return;
  const int bs = sub ? 4 : 8;
  const int nh = (width + (1 << fb_size_log2) - 1) >> fb_size_log2;
  const int f = (y >> fb_size_log2) * nh + (x >> fb_size_log2);
  const int X = src[y * stride + x];
  int out = X;
  const int bx = x & ~(bs - 1), by = y & ~(bs - 1);
  if (!allskip[f] && (!fb_on || fb_on[f]) && bi[((by << sub) / 4) * (width / 4) + ((bx << sub) / 4)].mode != 0) {
    // block-local clamping window (common/common_block.c:324-345): 2 samples beyond the block unless it lies on the
    // frame boundary
    const int sizex = min(width - bx, bs), sizey = min(height - by, bs);
    const int xmin = bx - (bx == 0 ? 0 : 2), ymin = by - (by == 0 ? 0 : 2);
    const int xmax = bx + sizex + (bx == width - sizex ? 0 : 2) - 1, ymax = by + sizey + (by == height - sizey ? 0 : 2) - 1;
    const S *r = src + y * stride;
    int A = src[max(ymin, y - 2) * stride + x], B = src[max(ymin, y - 1) * stride + x];
    int C = r[max(xmin, x - 2)], D = r[max(xmin, x - 1)], E = r[min(xmax, x + 1)], F = r[min(xmax, x + 2)];
    int G = src[min(ymax, y + 1) * stride + x], H = src[min(ymax, y + 2) * stride + x];
    out = X + clpf_sample(X, A, B, C, D, E, F, G, H, strength, (unsigned)damping);
  }
  dst[y * stride + x] = (S)out;
}
// single block, explicit boundary type (drop-in clpf_block4/8[_noclip])
template <class S>
__global__ void clpf_block_kernel(const S *src, S *dst, int sstride, int dstride, int x0, int y0, int sizex, int sizey, int bt, int strength, int damping) {
  const int xmin = x0 - !(bt & 1) * 2, ymin = y0 - !(bt & 4) * 2;
  const int xmax = x0 + sizex + !(bt & 2) * 2 - 1, ymax = y0 + sizey + !(bt & 8) * 2 - 1;
  for (int p = threadIdx.x; p < sizex * sizey; p += blockDim.x) {
    int y = y0 + p / sizex, x = x0 + p % sizex;
    int X = src[y * sstride + x];
    int d = clpf_sample(X, src[max(ymin, y - 2) * sstride + x], src[max(ymin, y - 1) * sstride + x], src[y * sstride + max(xmin, x - 2)],
                        src[y * sstride + max(xmin, x - 1)], src[y * sstride + min(xmax, x + 1)], src[y * sstride + min(xmax, x + 2)],
                        src[min(ymax, y + 1) * sstride + x], src[min(ymax, y + 2) * sstride + x], strength, (unsigned)damping);
    dst[y * dstride + x] = (S)(X + d);
  }
}
// detect_multi_clpf for every 8x8 block of a plane (enc/encode_block.c:2593-2624): one warp per block, 4 sums each
// (strength 0,1,2,4).  width,height = plane dimensions; skip lookup as in clpf_rdo (enc/encode_frame.c:566-569).
template <class S>
__global__ void __launch_bounds__(CTA_THREADS) clpf_detect_kernel(const S *rec, const S *org, int rstride, int ostride, int width, int height, const tb_blkinfo_t *bi,
                                                                  int luma_bw, int sub, int shift, int damping, int32_t *sums) {
  const int nbx = width >> 3, nby = height >> 3, lane = lane_id();
  for (int b = global_warp(); b < nbx * nby; b += total_warps()) {
    const int x0 = (b % nbx) * 8, y0 = (b / nbx) * 8;
    uint32_t s[4] = {0, 0, 0, 0};
    if (bi[((y0 << sub) / 4) * luma_bw + ((x0 << sub) / 4)].mode != 0) {
      for (int p = lane; p < 64; p += 32) {
        int y = y0 + (p >> 3), x = x0 + (p & 7);
        int O = org[y * ostride + x], X = rec[y * rstride + x];
        int A = rec[max(0, y - 2) * rstride + x], B = rec[max(0, y - 1) * rstride + x], C = rec[y * rstride + max(0, x - 2)],
            D = rec[y * rstride + max(0, x - 1)], E = rec[y * rstride + min(width - 1, x + 1)], F = rec[y * rstride + min(width - 1, x + 2)],
            G = rec[min(height - 1, y + 1) * rstride + x], H = rec[min(height - 1, y + 2) * rstride + x];
        s[0] += (uint32_t)((O - X) * (O - X));
#pragma unroll
        for (int t = 0; t < 3; t++) {
          int Y = X + clpf_sample(X, A, B, C, D, E, F, G, H, (1 << t) << shift, (unsigned)damping);
          s[t + 1] += (uint32_t)((O - Y) * (O - Y));
        }
      }
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
      uint32_t v = warp_sum(s[t]);
      if (lane == 0) sums[b * 4 + t] = (int32_t)(v >> (shift * 2));
    }
  }
}
// drop-in detect_clpf / detect_multi_clpf on one block (size x size), res[0..3]
template <class S>
__global__ void clpf_detect_block_kernel(const S *rec, const S *org, int x0, int y0, int width, int height, int ostride, int rstride, int strength, int shift,
                                         int size, int damping, int multi, uint32_t *res) {
  const int lane = lane_id();
  uint32_t s[4] = {0, 0, 0, 0};
  for (int p = lane; p < size * size; p += 32) {
    int y = y0 + p / size, x = x0 + p % size;
    int O = org[y * ostride + x], X = rec[y * rstride + x];
    int A = rec[max(0, y - 2) * rstride + x], B = rec[max(0, y - 1) * rstride + x], C = rec[y * rstride + max(0, x - 2)], D = rec[y * rstride + max(0, x - 1)],
        E = rec[y * rstride + min(width - 1, x + 1)], F = rec[y * rstride + min(width - 1, x + 2)], G = rec[min(height - 1, y + 1) * rstride + x],
        H = rec[min(height - 1, y + 2) * rstride + x];
    s[0] += (uint32_t)((O - X) * (O - X));
    if (multi) {
      for (int t = 0; t < 3; t++) {
        int Y = X + clpf_sample(X, A, B, C, D, E, F, G, H, (1 << t) << shift, (unsigned)damping);
        s[t + 1] += (uint32_t)((O - Y) * (O - Y));
      }
    } else {
      int Y = X + clpf_sample(X, A, B, C, D, E, F, G, H, strength, (unsigned)damping);
      s[1] += (uint32_t)((O - Y) * (O - Y));
    }
  }
  for (int t = 0; t < 4; t++) {
    uint32_t v = warp_sum(s[t]);
    if (lane == 0) res[t] = v;
  }
}

// ---- a19: CDEF -------------------------------------------------------------------------------------------------
// per 64x64 filter block all-skip flag (common/common_frame.c:809-823); width,height luma
__global__ void cdef_allskip_kernel(const tb_blkinfo_t *bi, int width, int height, uint8_t *allskip) {
  const int nh = (width + 63) >> 6, nv = (height + 63) >> 6;
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nh * nv) return;
  const int xoff = (f % nh) << 6, yoff = (f / nh) << 6;
  int all = 1;
  for (int m = 0; all && m < 8; m++)
    for (int n = 0; all && n < 8; n++) {
      int xpos = xoff + n * 8, ypos = yoff + m * 8;
      if (xpos < width && ypos < height) all &= bi[(ypos / 4) * (width / 4) + xpos / 4].mode == 0;
    }
  allskip[f] = (uint8_t)all;
}
// direction + variance of every 8x8 luma block in non-all-skip filter blocks; dirvar[(fb*2 + 0/1)*64 + m*8 + n]
template <class S>
__global__ void __launch_bounds__(CTA_THREADS) cdef_dir_kernel(const S *src, int stride, int width, int height, const uint8_t *allskip, int coeff_shift,
                                                               int32_t *dirvar) {
  const int nbx = (width + 7) >> 3, nby = (height + 7) >> 3, nh = (width + 63) >> 6;
  for (int b = global_warp(); b < nbx * nby; b += total_warps()) {
    const int bx = b % nbx, by = b / nbx, f = (by >> 3) * nh + (bx >> 3);
    if (allskip[f]) continue;
    int var;
    int dir = warp_cdef_find_dir<S>(src + by * 8 * stride + bx * 8, stride, coeff_shift, var);
    if (lane_id() == 0) {
      dirvar[(f * 2 + 0) * 64 + (by & 7) * 8 + (bx & 7)] = dir;
      dirvar[(f * 2 + 1) * 64 + (by & 7) * 8 + (bx & 7)] = var;
    }
  }
}
// out-of-place plane filter, one thread per sample.  width,height: LUMA dims; pw,ph: dims of this plane.
template <class S>
__global__ void cdef_plane_kernel(const S *src, S *dst, int stride, int width, int height, int pw, int ph, int sub, int plane, const tb_blkinfo_t *bi,
                                  const uint8_t *allskip, const int8_t *fb_pri, const int8_t *fb_sec, int pri_damping_f, int sec_damping_f,
                                  const int32_t *dirvar, int coeff_shift) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= pw || y >= ph) return;
  const int bslog = sub ? 2 : 3;
  const int lx = x << sub, ly = y << sub;  // luma coordinates
  const int nh = (width + 63) >> 6, f = (ly >> 6) * nh + (lx >> 6);
  const int X = src[y * stride + x];
  int out = X;
  const int n = (x >> bslog) & 7, m = (y >> bslog) & 7;  // block index inside the filter block
  if (!allskip[f] && bi[(((ly >> 6) * 64 + m * 8) >> 2) * (width >> 2) + (((lx >> 6) * 64 + n * 8) >> 2)].mode != 0) {
    const int pri = fb_pri[f], sec0 = fb_sec[f], sec = sec0 + (sec0 == 3);
    const int dir = dirvar[(f * 2 + 0) * 64 + m * 8 + n], var = dirvar[(f * 2 + 1) * 64 + m * 8 + n];
    const int adj = plane ? pri : adjust_strength(pri, var);
    int pd = pri_damping_f - (plane ? 1 : 0), sd = sec_damping_f - (plane ? 1 : 0);
    if (adj) pd = max(ilog2(adj), pd);
    const int ps = adj << coeff_shift, ss = sec << coeff_shift, d = pri ? dir : 0;
    pd += coeff_shift;
    sd += coeff_shift;
    // taps straight from the plane; outside the frame = CDEF_VERY_LARGE (common/common_frame.c:766-781)
    const int sel = (ps >> coeff_shift) & 1;
    const int pt[2] = {sel ? 3 : 4, sel ? 3 : 2}, st[2] = {2, 1};
    int mx = X, mn = X, sum = 0;
#pragma unroll
    for (int k = 0; k < 2; k++) {
      const int dirs[3] = {d, (d + 2) & 7, (d + 6) & 7};
#pragma unroll
      for (int g = 0; g < 3; g++) {
        const int dy = c_cdef_dy[dirs[g]][k], dx = c_cdef_dx[dirs[g]][k];
#pragma unroll
        for (int sgn = 0; sgn < 2; sgn++) {
          int yy = y + (sgn ? -dy : dy), xx = x + (sgn ? -dx : dx);
          int v = (yy < 0 || yy >= ph || xx < 0 || xx >= pw) ? 30000 : (int)src[yy * stride + xx];
          sum += (g == 0 ? pt[k] : st[k]) * constrain(v - X, g == 0 ? ps : ss, (unsigned)(g == 0 ? pd : sd));
          if (v != 30000) mx = max(mx, v);
          mn = min(mn, v);
        }
      }
    }
    sum = (int)(int16_t)sum;
    out = iclip(X + ((8 + sum - (sum < 0)) >> 4), mn, mx);
  }
  dst[y * stride + x] = (S)out;
}
// a19 (encoder): distortion table of cdef_search (enc/encode_frame.c:285-376).  One warp per (filter block, plane class,
// strength index): it filters every non-skip 8x8 block of the filter block with that strength and accumulates dist_8x8
// (double, round-to-nearest ops: no contraction) for full luma blocks or the plain SSE otherwise.  Reference quirks kept:
// chroma is filtered in 8x8 blocks whose skip flag / direction come from the top-left 4x4 entries of the block grid, and the
// secondary strength is used unadjusted (0..3).
__constant__ int8_t c_priconv[3][16] = {{0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {0, 1, 2, 3, 5, 7, 10, 13, 0, 0, 0, 0, 0, 0, 0, 0}, {0, 1, 3, 6, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}};
template <class S>
__global__ void __launch_bounds__(CTA_THREADS) cdef_search_kernel(const S *recY, const S *recU, const S *recV, const S *orgY, const S *orgU, const S *orgV, int sy, int sc,
                                                                  int width, int height, const tb_blkinfo_t *bi, const uint8_t *allskip, const int32_t *dirvar, int speed,
                                                                  int total, int pri_damping, int coeff_shift, unsigned long long *mse) {
  const int nh = (width + 63) >> 6, nv = (height + 63) >> 6, nfb = nh * nv, lane = lane_id();
  const int units = nfb * 2 * total;
  for (int u = global_warp(); u < units; u += total_warps()) {
    const int gi = u % total, cls = (u / total) & 1, fb = u / (2 * total);
    if (allskip[fb]) {
      if (lane == 0) mse[(size_t)cls * nfb * 64 + fb * 64 + gi] = 0;
      continue;
    }
    const int l = fb % nh, k = fb / nh, xoff = l << 6, yoff = k << 6;
    int h = min(height, (k + 1) << 6) & 63, w = min(width, (l + 1) << 6) & 63;
    h += !h << 6;
    w += !w << 6;
    const int pri = c_priconv[speed][gi >> 2], sec = gi & 3;
    unsigned long long acc = 0;
    for (int plane = cls ? 1 : 0; plane <= (cls ? 2 : 0); plane++) {
      const int sub = plane != 0, st = plane ? sc : sy, pw = width >> sub, ph = height >> sub;
      const S *src = plane ? (plane == 1 ? recU : recV) : recY, *org = plane ? (plane == 1 ? orgU : orgV) : orgY;
      const int nbm = (h + 7) >> (3 + sub), nbn = (w + 7) >> (3 + sub);
      for (int b = 0; b < nbm * nbn; b++) {
        const int m = b / nbn, n = b - m * nbn;
        const int xpos = (xoff >> sub) + n * 8, ypos = (yoff >> sub) + m * 8;
        const int sizex = min(pw - xpos, 8), sizey = min(ph - ypos, 8);
        if (bi[(((yoff + m * 8) >> 2)) * (width >> 2) + ((xoff + n * 8) >> 2)].mode == 0) continue;
        const int dir = dirvar[(fb * 2 + 0) * 64 + m * 8 + n], var = dirvar[(fb * 2 + 1) * 64 + m * 8 + n];
        const int adj = plane ? pri : adjust_strength(pri, var);
        int pd = pri_damping - (plane ? 1 : 0), sd = pri_damping - (plane ? 1 : 0);
        if (adj) pd = max(ilog2(adj), pd);
        const int ps = adj << coeff_shift, ss = sec << coeff_shift, d = pri ? dir : 0;
        pd += coeff_shift;
        sd += coeff_shift;
        const int sel = (ps >> coeff_shift) & 1;
        const int pt[2] = {sel ? 3 : 4, sel ? 3 : 2}, stp[2] = {2, 1};
        unsigned long long s_s = 0, s_d = 0, s_s2 = 0, s_d2 = 0, s_sd = 0, sse = 0;
        for (int p = lane; p < sizex * sizey; p += 32) {
          const int i = p / sizex, j = p - i * sizex, x = xpos + j, y = ypos + i;
          const int X = src[y * st + x];
          int mx = X, mn = X, sum = 0;
#pragma unroll
          for (int t = 0; t < 2; t++) {
            const int dirs3[3] = {d, (d + 2) & 7, (d + 6) & 7};
#pragma unroll
            for (int g = 0; g < 3; g++) {
              const int dy = c_cdef_dy[dirs3[g]][t], dx = c_cdef_dx[dirs3[g]][t];
#pragma unroll
              for (int sgn = 0; sgn < 2; sgn++) {
                int yy = y + (sgn ? -dy : dy), xx = x + (sgn ? -dx : dx);
                int v = (yy < 0 || yy >= ph || xx < 0 || xx >= pw) ? 30000 : (int)src[yy * st + xx];
                sum += (g == 0 ? pt[t] : stp[t]) * constrain(v - X, g == 0 ? ps : ss, (unsigned)(g == 0 ? pd : sd));
                if (v != 30000) mx = max(mx, v);
                mn = min(mn, v);
              }
            }
          }
          sum = (int)(int16_t)sum;
          const int F = iclip(X + ((8 + sum - (sum < 0)) >> 4), mn, mx);
          const int Oo = org[y * st + x];
          s_s += (unsigned)Oo; s_d += (unsigned)F; s_s2 += (unsigned)(Oo * Oo); s_d2 += (unsigned)(F * F); s_sd += (unsigned)(Oo * F);
          sse += (unsigned)((F - Oo) * (F - Oo));
        }
        if (plane || sizex != 8 || sizey != 8) {
          acc += warp_sum64(sse);
        } else {
          s_s = warp_sum64(s_s); s_d = warp_sum64(s_d); s_s2 = warp_sum64(s_s2); s_d2 = warp_sum64(s_d2); s_sd = warp_sum64(s_sd);
          // dist_8x8 (enc/encode_frame.c:194-221), ISO-C evaluation order with explicitly rounded double operations
          const unsigned long long svar = s_s2 - ((s_s * s_s + 32) >> 6), dvar = s_d2 - ((s_d * s_d + 32) >> 6);
          const double a = __dmul_rn(__ull2double_rn(s_d2 + s_s2 - 2 * s_sd), 0.5);
          const double bb = __dmul_rn(a, __ull2double_rn(svar + dvar + (unsigned long long)(400 << 2 * coeff_shift)));
          const double den = __dsqrt_rn(__dadd_rn((double)(20000 << 4 * coeff_shift), __dmul_rn(__ull2double_rn(svar), __ull2double_rn(dvar))));
          acc += (unsigned long long)floor(__dadd_rn(0.5, __ddiv_rn(bb, den)));
        }
      }
    }
    if (lane == 0) mse[(size_t)cls * nfb * 64 + fb * 64 + gi] = acc;
  }
}

// drop-in cdef_filter_block_simd on a staged uint16 tile
__global__ void cdef_block_kernel(uint8_t *dst8, uint16_t *dst16, int dstride, const uint16_t *in, int sstride, int pri, int sec, int dir, int pd, int sd, int bsize,
                                  int coeff_shift) {
  for (int p = threadIdx.x; p < bsize * bsize; p += blockDim.x) {
    int i = p / bsize, j = p % bsize;
    int y = cdef_sample(in + i * sstride + j, sstride, pri, sec, dir, pd, sd, coeff_shift);
    if (dst8) dst8[i * dstride + j] = (uint8_t)y;
    else dst16[i * dstride + j] = (uint16_t)y;
  }
}
template <class S> __global__ void cdef_dir_block_kernel(const S *img, int stride, int coeff_shift, int32_t *res) {
  int var;
  int dir = warp_cdef_find_dir<S>(img, stride, coeff_shift, var);
  if (lane_id() == 0) { res[0] = dir; res[1] = var; }
}

// ---- a20/a21: padding, reference copy, down-scaling -----------------------------------------------------------
// dst(padded plane) = src[clamp]: one pass writes the visible area and the replicated border
// (common/common_frame.c:657-764).  dst, src point at sample (0,0).
template <class S>
__global__ void pad_copy_kernel(S *dst, int ds, const S *src, int ss, int w, int h, int pad_hor, int pad_ver, int border_only) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x - pad_hor, y = blockIdx.y * blockDim.y + threadIdx.y - pad_ver;
  if (x >= w + pad_hor || y >= h + pad_ver) return;
  const bool inside = x >= 0 && x < w && y >= 0 && y < h;
  if (border_only && inside) return;
  dst[y * ds + x] = src[iclip(y, 0, h - 1) * ss + iclip(x, 0, w - 1)];
}
template <class S> __global__ void scale_down_kernel(const S *in, int si, S *out, int so, int wo, int ho) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= wo || y >= ho) return;
  const S *p = in + 2 * y * si + 2 * x;
  out[y * so + x] = (S)((up2(p[0], p[si]) + up2(p[1], p[si + 1])) >> 1);
}

}  // namespace tb
