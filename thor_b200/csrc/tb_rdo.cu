// tb_rdo.cu — SURVEY.md §8f.1: the reference's per-super-block RD loop resident on the GPU.
//
// tb_rdo_encode_frames() (include/thor_b200.h) uploads the source frames and their padded reference frames, runs rdo_batch_kernel —
// persistent CTAs that draw READY super blocks from the rows of every frame of the batch (row r may process super block c when row r-1
// has published c+2 super blocks: left, up-left, up, up-right neighbours; frames are independent) — and downloads the decisions
// (reconstruction, per-4x4 block state, the leaf list of every super block with its coefficients).
// The control flow is tb_rdo.h (shared with the CPU host check that pins it against the reference); this file supplies its backend:
// the warp-cooperative primitives of tb_device.cuh / tb_kernels.cuh, i.e. the same device routines the batched tb_* entry points
// and the drop-in symbols use (parity-tested against the oracle one by one in tests/test_gpu_parity.py).
//
// This is a separate translation unit because two load policies differ from the batched kernels:
//   TB_LDG -> plain load: the "original" of a search can be a scratch block this CTA wrote a moment ago (bipred target 2*org - pred),
//             so the read-only (non-coherent) path must not be used;
//   TB_LDF -> __ldcg: reconstructed samples and block state of the neighbouring super blocks were written by OTHER CTAs during this
//             launch; L1 is not coherent across SMs and a line can straddle two super blocks, so those loads bypass L1.
// The device code of this unit lives in its own namespace (the headers define __constant__ tables).
#define TB_LDG(p) (*(p))
#define TB_LDF(p) __ldcg(p)
#define TB_ROLL _Pragma("unroll 1")  // loops stay loops: the kernel is bound by instruction fetch, not by loop overhead
#define TB_ME_STAGE_PROF 1  // cycles per search stage (telescope, candidates, hexagon, half-pel, quarter-pel) of blocks <= 16 in the kernel's counters
#define TB_SAD_ROWS 1  // integer-position SADs of blocks >= 32 bytes wide: lanes along the row (multi_sad_rows)
#define tb tb_rdo_tu
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include "tb_kernels.cuh"
#include "tb_rdo.h"

using namespace tb;
using namespace tbr;

namespace {

// per-primitive cycle counters (TB_RDO_PROF=1): which part of the RD loop the warp spends its time in
enum { PF_INTERP, PF_ME, PF_MEBI, PF_TX, PF_BITS, PF_SSD, PF_INTRA, PF_COPY, PF_ES, PF_WAIT, PF_TOTAL, PF_N };
// always-on work counters (SURVEY.md §8d algorithmic samples of what the RD loop actually executed: the loop is data dependent) behind the cycle counters:
// searches, integer block SADs, sub-pel probes, search samples, predictions, prediction samples, transform chains, chain samples, intra predictions, intra samples,
// SSD/SAD samples, super blocks
enum { ST_ME = PF_N, ST_ME_INT, ST_ME_SUB, ST_ME_SAMPLES, ST_IP, ST_IP_SAMPLES, ST_TX, ST_TX_SAMPLES, ST_INTRA, ST_INTRA_SAMPLES, ST_SSD_SAMPLES, ST_SB,
       ST_ME_SZ /* cycles of searches by coding-block size 8..128 */, ST_TX_SZ = ST_ME_SZ + 5 /* chains by transform size 4..128 */, ST_IP_SZ = ST_TX_SZ + 6 /* predictions by width 4..128 */,
       ST_PH = ST_IP_SZ + 6 /* wall cycles of warp 0 by decision phase (tb_rdo.h PH_*) */, ST_MESTAGE = ST_PH + tbr::PH_N /* search stages, coding blocks <= 16 */,
       ST_X = ST_MESTAGE + 5 /* search phase of a block decision: warp 0 {own searches, -, barrier wait}, warp nw-1 {-, intra items, barrier wait} */, ST_END = ST_X + 6 };
struct Prof {
  long long *acc;
  int k, k2;
  long long t0;
#ifdef __CUDA_ARCH__
  __device__ __forceinline__ Prof(long long *a, int kk, int kk2 = -1) : acc(a), k(kk), k2(kk2), t0(clock64()) {}
  __device__ __forceinline__ ~Prof() { const long long d = clock64() - t0; acc[k] += d; if (k2 >= 0) acc[k2] += d; }
#else
  Prof(long long *a, int kk, int kk2 = -1) : acc(a), k(kk), k2(kk2), t0(0) {}
#endif
};

static_assert(ST_END == TB_RDO_NSTATS, "tb_rdo_batch_stats layout");
constexpr int RDO_MAX_WARPS = 16;
// per-CTA: tables and the exchange area of the SPMD control flow (tb_rdo.h)
struct RdoCta {
  alignas(16) int8_t tab8[TX_TABLE_BYTES];       // int8 DCT matrices (plain, transposed) + 16x16 zig-zag table
  alignas(16) int16_t tab16[DCT_TAB_SIZE];       // int16 DCT matrices (warp_fwd_transform of the early-skip test)
  uint32_t x_cost[RDO_MAX_WARPS];
  int x_idx[RDO_MAX_WARPS];
  uint32_t x_rng[RDO_MAX_WARPS][2];
  int x_flag[RDO_MAX_WARPS];
  tb_mv_t x_mv[TB_RDO_MAX_REF][16];
  uint32_t x_sad[TB_RDO_MAX_REF];
  alignas(16) int x_buf[32];
  int x_queue[4];
  int sel;
};
// per-warp scratch
template <class S> struct RdoShared {
  long long prof[ST_END];
  long long t_mark, t_mark2;
  alignas(16) unsigned char jobs[12 * 64];  // tx_multi: the chains' parameters
  TxScratch sc;
  alignas(16) int16_t blk16[256];                // early skip: averaged residual / chroma residual
  alignas(16) int16_t out16[256];                // transform output of the early-skip test; coefficient scan for the bit count
  alignas(16) S left[256], top[256], filt[4 * 128 + 4];
  tb_txfm_result_t res;
};

template <class S> struct DevBackend {
  const FrameCtx<S> *F;
  RdoShared<S> *sh;  // this warp's scratch
  RdoCta *cta;
  int nw, wid;

  // ---- SPMD over the warps of the CTA (tb_rdo.h): every warp reaches every CTA barrier (the control flow is replicated)
  __device__ __forceinline__ int warp() const { return wid; }
  __device__ __forceinline__ bool mine(int k) const { return (k % nw) == wid; }
  __device__ void cta_sync() const { __threadfence(); __syncthreads(); }
  __device__ __forceinline__ int nwarps() const { return nw; }
  __device__ __noinline__ void queue_reset() const {
    __syncthreads();
    if (threadIdx.x < 4) cta->x_queue[threadIdx.x] = 0;
    __syncthreads();
  }
  __device__ int next(int q) const {  // shared counter: every lane of the warp receives the drawn value
    int v = 0;
    if ((threadIdx.x & 31) == 0) v = atomicAdd(&cta->x_queue[q], 1);
    return __shfl_sync(FULL, v, 0);
  }
  __device__ __noinline__ void copy_words(void *dst, const void *src, int nwords) const {
    __syncwarp();
    for (int k = threadIdx.x & 31; k < nwords; k += 32) ((int *)dst)[k] = ((const int *)src)[k];
    __syncwarp();
  }
  __device__ __forceinline__ void mark2(int k) const {  // per-warp timers of the search phase, kept for warp 0 and the last warp
    if ((wid == 0 || wid == nw - 1) && (threadIdx.x & 31) == 0) {
      const long long t = clock64();
      if (k >= 0) sh->prof[ST_X + (wid == 0 ? 0 : 3) + k] += t - sh->t_mark2;
      sh->t_mark2 = t;
    }
  }
  __device__ __forceinline__ void mark(int k) const {
    if (wid == 0 && (threadIdx.x & 31) == 0) { const long long t = clock64(); sh->prof[ST_PH + k] += t - sh->t_mark; sh->t_mark = t; }
  }
  __device__ void put_me(int ref, const Mv *mv16, uint32_t sad) const {
    if ((threadIdx.x & 31) < 16) cta->x_mv[ref][threadIdx.x & 31] = mv16[threadIdx.x & 31];
    if ((threadIdx.x & 31) == 0) cta->x_sad[ref] = sad;
  }
  __device__ void get_me(int ref, Mv *mv16, uint32_t *sad) const {  // every lane fills its own (replicated) copy
#pragma unroll
    for (int k = 0; k < 16; k++) mv16[k] = cta->x_mv[ref][k];
    *sad = cta->x_sad[ref];
  }
  __device__ __noinline__ int reduce_best(uint32_t *cost, int *idx) const {
    if ((threadIdx.x & 31) == 0) { cta->x_cost[wid] = *cost; cta->x_idx[wid] = *idx; }
    __syncthreads();
    int w = 0;
    for (int k = 1; k < nw; k++)
      if (cta->x_cost[k] < cta->x_cost[w] || (cta->x_cost[k] == cta->x_cost[w] && cta->x_idx[k] < cta->x_idx[w])) w = k;
    *cost = cta->x_cost[w]; *idx = cta->x_idx[w];
    __syncthreads();
    return w;
  }
  __device__ __noinline__ void bcast(void *p, int nbytes, int owner) const {  // p: per-thread (replicated) object, multiple of 4 bytes, <= 128
    int *q = (int *)p;
    if (wid == owner && (threadIdx.x & 31) == 0)
      TB_ROLL
      for (int k = 0; k < nbytes / 4; k++) cta->x_buf[k] = q[k];
    __syncthreads();
    if (wid != owner)
      TB_ROLL
      for (int k = 0; k < nbytes / 4; k++) q[k] = cta->x_buf[k];
    __syncthreads();
  }
  __device__ __noinline__ void reduce_range(uint32_t *worst, uint32_t *best) const {
    if ((threadIdx.x & 31) == 0) { cta->x_rng[wid][0] = *worst; cta->x_rng[wid][1] = *best; }
    __syncthreads();
    for (int k = 0; k < nw; k++) { *worst = max(*worst, cta->x_rng[k][0]); *best = min(*best, cta->x_rng[k][1]); }
    __syncthreads();
  }
  __device__ __noinline__ int reduce_or(int f) const {
    if ((threadIdx.x & 31) == 0) cta->x_flag[wid] = f;
    __syncthreads();
    int r = 0;
    for (int k = 0; k < nw; k++) r |= cta->x_flag[k];
    __syncthreads();
    return r;
  }

  __device__ __forceinline__ int lane() const { return threadIdx.x & 31; }
#define PROF(k) Prof prof__(sh->prof, k)
#define PROF2(k, k2) Prof prof__(sh->prof, k, k2)
  __device__ __forceinline__ void sync() const { __syncwarp(); }

  __device__ __noinline__ tb_rdo_blk_t ld_blk(const tb_rdo_blk_t *p) const {
    // 20 bytes, 4-byte aligned; written by another CTA earlier in this launch -> L2
    const int *q = (const int *)p;
    int w[5];
#pragma unroll
    for (int k = 0; k < 5; k++) w[k] = __ldcg(q + k);
    tb_rdo_blk_t b;
    memcpy(&b, w, sizeof(b));
    return b;
  }
  __device__ void clip_mv(Mv &mv, int ypos, int xpos, int fw, int fh, int bw, int bh, int sign) const {
    int x = mv.x, y = mv.y;
    tb::clip_mv(x, y, ypos, xpos, fw, fh, bw, bh, sign);
    mv.x = (int16_t)x; mv.y = (int16_t)y;
  }
  // prediction of one block; widths that are not powers of two (rectangular blocks at the right frame edge) take the per-sample form
  __device__ __noinline__ void interp_any(S *dst, int ds, const S *ref, int rs, int w, int h, Mv mv, int sign, int chroma, int bip, int pw, int ph, int xpos, int ypos) const {
    PROF2(PF_INTERP, ST_IP_SZ + min(5, max(0, ilog2(max(w, h)) - 2)));
    if (lane() == 0) { sh->prof[ST_IP] += 1; sh->prof[ST_IP_SAMPLES] += (xf_any(mv, chroma) ? (w + 5) * (h + 5) : w * h) + w * h; }
    sync();
    if (!(w & (w - 1))) warp_interp<S>(dst, ds, ref, rs, w, h, mv.x, mv.y, sign, chroma, bip, pw, ph, xpos, ypos, F->bitdepth);
    else {
      int hi, vi, xf, yf;
      split_mv(mv.x, mv.y, sign, chroma ? 3 : 2, pw, ph, xpos, ypos, w, h, hi, vi, xf, yf);
      const S *ip = ref + vi * rs + hi;
      const int maxv = (1 << F->bitdepth) - 1;
      TB_ROLL
      for (int p = lane(); p < w * h; p += 32) {
        const int row = p / w, col = p - row * w;
        const S *q = ip + row * rs + col;
        int v;
        if (xf == 0 && yf == 0) v = q[0];
        else v = chroma ? chroma_sample<S>(q, rs, xf, yf, maxv) : luma_sample<S>(q, rs, xf, yf, bip, maxv);
        dst[row * ds + col] = (S)v;
      }
    }
    sync();
  }
  __device__ __forceinline__ static int xf_any(Mv mv, int chroma) { return chroma ? ((mv.x | mv.y) & 7) : ((mv.x | mv.y) & 3); }
  __device__ void interp_luma(S *dst, int ds, const S *ref, int rs, int w, int h, Mv mv, int sign, int bip, int pw, int ph, int xpos, int ypos) const {
    interp_any(dst, ds, ref, rs, w, h, mv, sign, 0, bip, pw, ph, xpos, ypos);
  }
  __device__ void interp_chroma(S *dst, int ds, const S *ref, int rs, int w, int h, Mv mv, int sign, int pw, int ph, int xc, int yc) const {
    interp_any(dst, ds, ref, rs, w, h, mv, sign, 1, 0, pw, ph, xc, yc);
  }
  __device__ __noinline__ void avg(S *dst, const S *a, const S *b, int stride, int w, int h) const {
    PROF(PF_COPY);
    sync();
    TB_ROLL
    for (int p = lane(); p < w * h; p += 32) {
      const int row = p / w, col = p - row * w, o = row * stride + col;
      dst[o] = (S)(((int)a[o] + (int)b[o]) >> 1);
    }
    sync();
  }
  __device__ __noinline__ void sat2ab(S *dst, const S *org, int os, const S *pred, int size) const {
    PROF(PF_COPY);
    const int maxv = (1 << F->bitdepth) - 1, ls = ilog2(size);
    sync();
    TB_ROLL
    for (int p = lane(); p < size * size; p += 32) {
      const int row = p >> ls, col = p & (size - 1);
      dst[p] = (S)sat_px(2 * (int)org[row * os + col] - (int)pred[p], maxv);
    }
    sync();
  }
  __device__ __noinline__ void copy(S *dst, int ds, const S *src, int ss, int w, int h) const {
    PROF(PF_COPY);
    sync();
    TB_ROLL
    for (int p = lane(); p < w * h; p += 32) {
      const int row = p / w, col = p - row * w;
      dst[row * ds + col] = src[row * ss + col];
    }
    sync();
  }
  __device__ __noinline__ void copy_coeff(int16_t *dst, const int16_t *src) const {
    PROF(PF_COPY);
    sync();
    TB_ROLL
    for (int p = lane(); p < 1024 / 4; p += 32) ((uint2 *)dst)[p] = ((const uint2 *)src)[p];
    sync();
  }
  __device__ __noinline__ void intra_predict(S *dst, int ds, const S *recf, int rfs, const S *rblock, int rbs, int i, int j, int ypos, int xpos, int size, int ur, int dl, int tbs,
                                int mode) const {
    PROF(PF_INTRA);
    if (lane() == 0) { sh->prof[ST_INTRA] += 1; sh->prof[ST_INTRA_SAMPLES] += 4 * size + size * size; }
    sync();
    S tl;
    warp_make_top_and_left<S>(sh->left, sh->top, tl, recf, rfs, rblock, rbs, i, j, ypos, xpos, size, ur, dl, tbs, F->bitdepth);
    sync();
    if (mode == 10) warp_intra_pred<S>(sh->left, sh->top, tl, 1, 1, size, dst, ds, 0, F->bitdepth, sh->filt);  // DC from (left, top) as gathered
    else warp_intra_pred<S>(sh->left, sh->top, tl, ypos + i, xpos + j, size, dst, ds, mode, F->bitdepth, sh->filt);
    sync();
  }
  __device__ __noinline__ void cfl(const S *y, S *u, S *v, const S *ry, int n, int cstride, int stride) const {
    PROF(PF_INTRA);
    sync();
    warp_cfl<S>(y, u, v, ry, n, cstride, stride, 1, F->bitdepth);
    sync();
  }
  __device__ __noinline__ int tx_chain(const S *orig, int os, const S *pred, int ps, S *rec, int rs, int16_t *cq, int size, int qp, int coeff_type, int fast) const {
    int cbp;
    if (size < 16) {  // 4x4 / 8x8: the loop form below, one chain
      tbr::TxJob<S> j;
      j.orig = orig; j.pred = pred; j.rec = rec; j.cq = cq; j.os = os; j.ps = ps; j.rs = rs; j.size = size; j.qp = qp; j.coeff_type = coeff_type; j.fast = fast;
      tx_multi(&j, 1, &cbp);
      return cbp;
    }
    PROF2(PF_TX, ST_TX_SZ + ilog2(size) - 2);
    if (lane() == 0) { sh->prof[ST_TX] += 1; sh->prof[ST_TX_SAMPLES] += 3 * size * size; }
    sync();
    tb_txfm_item_t q;
    q.orig = orig; q.pred = pred; q.rec = rec; q.coeffq = cq; q.ostride = os; q.pstride = ps; q.rstride = rs;
    q.size = (uint8_t)size; q.qp = (uint8_t)qp; q.coeff_type = (uint8_t)coeff_type; q.fast = (uint8_t)(fast ? TB_TXFM_FAST : 0);
    tx_big_chain<S, 1>(q, F->bitdepth, sh->sc, nullptr, cta->tab8, cta->tab8 + DCT_TAB8_SIZE, nullptr, nullptr, &sh->res);
    sync();
    cbp = sh->res.cbp;
    sync();
    return cbp;
  }
  // <= 12 chains of 4x4 / 8x8 transform blocks (residual -> DCT -> quantiser -> dequantiser -> inverse DCT -> reconstruction, the arithmetic of
  // common/transform.c:245-308, 411-494, enc/encode_block.c:84-171, common/common_block.c:45-83), all of them together on the warp.  Written as LOOPS over
  // (chain, element) work items dealt to the lanes: the RD loop is bound by instruction fetch (ncu: 19 stalled warps per issued instruction wait for
  // instructions), so a few hundred instructions that stay in the instruction cache beat the unrolled one-thread-per-chain forms (5.6 k instructions
  // streamed from L2 per call).  Tiles of 64 int16 per chain in the warp's scratch; the quantiser's level-mode walk is sequential: one lane per chain.
  __device__ __noinline__ void tx_multi(const tbr::TxJob<S> *jobs, int n, int *bit) const {
    PROF2(PF_TX, ST_TX_SZ + ilog2(jobs[0].size) - 2);
    const int l = lane();
    if (l == 0)
      TB_ROLL
      for (int k = 0; k < n; k++) { sh->prof[ST_TX] += 1; sh->prof[ST_TX_SAMPLES] += 3 * jobs[k].size * jobs[k].size; }
    int16_t *A = sh->sc.in, *B = sh->sc.in + 768;  // 12 tiles of 64 each
    // chain parameters in shared memory (per warp): the loops index them by chain
    tbr::TxJob<S> *J = (tbr::TxJob<S> *)sh->jobs;
    sync();
    if (l < n) J[l] = jobs[l];
    sync();
    const int bd = F->bitdepth, maxv = (1 << bd) - 1;
    // (1) residual -> A[k][i * N + j]
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63;
      const tbr::TxJob<S> &q = J[k];
      const int N = q.size, ln = N == 8 ? 3 : 2;
      if (e < N * N) { const int i = e >> ln, j = e & (N - 1); A[w] = (int16_t)((int)q.orig[i * q.os + j] - (int)q.pred[i * q.ps + j]); }
    }
    sync();
    // (2) forward, first dimension: B[k][i][j] = (sum_t M[i][t] * A[k][j][t] + add1) >> shift1
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63, N = J[k].size, ln = N == 8 ? 3 : 2;
      if (e < N * N) {
        const int i = e >> ln, j = e & (N - 1);
        const int16_t *M = cta->tab16 + (N == 8 ? 16 : 0) + (i << ln), *a = A + (k << 6) + (j << ln);
        int sum = 0;
        TB_ROLL
        for (int t = 0; t < N; t++) sum += (int)M[t] * (int)a[t];
        const int shift1 = ln + bd - 8;
        B[w] = (int16_t)((sum + (1 << (shift1 - 1))) >> shift1);
      }
    }
    sync();
    // (3) forward, second dimension: A[k][i][j] = (sum_t M[i][t] * B[k][j][t] + add2) >> shift2   (coefficients, raster)
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63, N = J[k].size, ln = N == 8 ? 3 : 2;
      int v = 0;
      if (e < N * N) {
        const int i = e >> ln, j = e & (N - 1);
        const int16_t *M = cta->tab16 + (N == 8 ? 16 : 0) + (i << ln), *b = B + (k << 6) + (j << ln);
        int sum = 0;
        TB_ROLL
        for (int t = 0; t < N; t++) sum += (int)M[t] * (int)b[t];
        const int shift2 = ln + 5;
        v = (sum + (1 << (shift2 - 1))) >> shift2;
      }
      if (e < N * N) A[w] = (int16_t)v;  // A was consumed by (2)
    }
    sync();
    // (4) zig-zag scan order -> B[k][pos]
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63, N = J[k].size, ln = N == 8 ? 3 : 2;
      if (e < N * N) B[(k << 6) + zigzag_index(e >> ln, e & (N - 1), N)] = A[w];
    }
    sync();
    // (5) quantiser (sequential level-mode walk), lane k on chain k: levels in scan order -> B[k][pos] in place; cbp
    int cbp = 0;
    if (l < n) {
      const tbr::TxJob<S> &q = J[l];
      const int N = q.size, nq = N * N, intra = (q.coeff_type >> 1) & 1, scale = c_quant[q.qp % 6], shift2 = 21 - (N == 8 ? 3 : 2) + q.qp / 6;
      int16_t *sc_ = B + (l << 6);
      const int offset = (intra ? 38 : -26) * (1 << (shift2 - 8));
      int level = 0, pos = nq - 1;
      while (level == 0 && pos >= 0) {
        const int v = iabs((int)sc_[pos]) * scale + offset;  // < 2^31: |c| <= 32768, scale <= 26214
        level = iabs(v) >> shift2;
        pos--;
      }
      const int last_pos = level ? pos + 1 : pos;
      const int off0 = (intra ? 102 : 51) << (shift2 - 8), off1 = (intra ? 115 : 90) << (shift2 - 8);
      int level_mode = 1;
      TB_ROLL
      for (pos = 0; pos <= last_pos; pos++) {
        const int c = sc_[pos];
        const unsigned ac = (unsigned)scale * (unsigned)iabs(c);
        const int level0 = (int)(ac >> shift2);
        const int lev = (int)((ac + (unsigned)((level0 > (1 - level_mode)) ? off1 : off0)) >> shift2);
        sc_[pos] = (int16_t)(c < 0 ? -lev : lev);
        cbp |= lev != 0;
        if (level_mode) { if (lev == 0) level_mode = 0; }
        else if (lev > 1) level_mode = 1;
      }
      TB_ROLL
      for (pos = last_pos + 1; pos < nq; pos++) sc_[pos] = 0;
    }
    sync();
    const unsigned nzmask = __ballot_sync(FULL, cbp != 0);
    // (6) quantised coefficients, raster: to the caller's buffer (reference layout) and, dequantised, to A[k] (dequantize(), common/common_block.c:45)
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63;
      const tbr::TxJob<S> &q = J[k];
      const int N = q.size, ln = N == 8 ? 3 : 2;
      if (e < N * N) {
        const int c = B[(k << 6) + zigzag_index(e >> ln, e & (N - 1), N)];
        q.cq[e] = (int16_t)c;
        const int lshift = q.qp / 6, rshift = ln - 1, dscale = c_dequant[q.qp % 6];
        A[w] = lshift >= rshift ? (int16_t)((c * dscale) << (lshift - rshift)) : (int16_t)((c * dscale + (1 << (rshift - lshift - 1))) >> (rshift - lshift));
      }
    }
    sync();
    // (7) inverse, first dimension: B[k][i][j] = sat16((sum_t M[t][j] * A[k][t][i] + 64) >> 7)
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63, N = J[k].size, ln = N == 8 ? 3 : 2;
      if (e < N * N && ((nzmask >> k) & 1)) {
        const int i = e >> ln, j = e & (N - 1);
        const int16_t *M = cta->tab16 + (N == 8 ? 16 : 0), *a = A + (k << 6);
        int o = 0;
        TB_ROLL
        for (int t = 0; t < N; t++) o += (int)M[(t << ln) + j] * (int)a[(t << ln) + i];
        o = (o + 64) >> 7;
        B[w] = (int16_t)iclip(o, -32768, 32767);
      }
    }
    sync();
    // (8) inverse, second dimension + reconstruction: rec = clip(pred + sat16((sum_t M[t][j] * B[k][t][i] + round) >> (20 - bitdepth))); no coefficient: rec = pred
    TB_ROLL
    for (int w = l; w < n * 64; w += 32) {
      const int k = w >> 6, e = w & 63;
      const tbr::TxJob<S> &q = J[k];
      const int N = q.size, ln = N == 8 ? 3 : 2;
      if (e < N * N) {
        const int i = e >> ln, j = e & (N - 1);
        int v = (int)q.pred[i * q.ps + j];
        if ((nzmask >> k) & 1) {
          const int16_t *M = cta->tab16 + (N == 8 ? 16 : 0), *b = B + (k << 6);
          int o = 0;
          TB_ROLL
          for (int t = 0; t < N; t++) o += (int)M[(t << ln) + j] * (int)b[(t << ln) + i];
          const int sh2 = 20 - bd;
          o = (o + (1 << (sh2 - 1))) >> sh2;
          v = sat_px(v + iclip(o, -32768, 32767), maxv);
        }
        q.rec[i * q.rs + j] = (S)v;
      }
    }
    sync();
    for (int k = 0; k < n; k++) bit[k] = (nzmask >> k) & 1;
  }
  __device__ __noinline__ int coeff_bits(const int16_t *cq, int size, int type) const {
    PROF(PF_BITS);
    const int qs = min(size, 16), nq = qs * qs, lq = ilog2(qs);
    sync();
    TB_ROLL
    for (int p = lane(); p < nq; p += 32) sh->out16[zigzag_index(p >> lq, p & (qs - 1), qs)] = cq[p];
    sync();
    const int bits = warp_coeff_bits(sh->out16, nq, size, type);
    sync();
    return bits;
  }
  __device__ __noinline__ uint64_t ssd(const S *a, int as, const S *b, int bs, int w, int h) const {
    PROF(PF_SSD);
    if (lane() == 0) sh->prof[ST_SSD_SAMPLES] += 2 * w * h;
    sync();
    if (!(w & (w - 1))) return warp_ssd<S>(a, as, b, bs, w, h);
    uint64_t acc = 0;
    TB_ROLL
    for (int p = lane(); p < w * h; p += 32) {
      const int row = p / w, col = p - row * w, d = (int)a[row * as + col] - (int)b[row * bs + col];
      acc += (uint64_t)(uint32_t)(d * d);
    }
    return warp_sum64(acc);
  }
  __device__ __noinline__ unsigned sad(const S *a, int as, const S *b, int bs, int w, int h) const {
    PROF(PF_SSD);
    if (lane() == 0) sh->prof[ST_SSD_SAMPLES] += 2 * w * h;
    sync();
    return warp_sad<S>(a, as, b, bs, w, h);
  }
  __device__ __noinline__ int me(const S *org, int os, const S *ref, int rs, int size, int w, int h, Mv *mv, Mv mvc, Mv mvp, double lambda, int sign, int xpos, int ypos, const Mv *cand,
                    int ncand) const {
    PROF2(PF_ME, ST_ME_SZ + ilog2(size) - 3);
    sync();
    MeCtx c;
    c.size = size; c.width = w; c.height = h; c.sign = sign; c.s = sign ? -1 : 1; c.xpos = xpos; c.ypos = ypos; c.fw = F->width; c.fh = F->height;
    c.bitdepth = F->bitdepth; c.speed = F->speed; c.bip = F->enable_bipred; c.mvpx = mvp.x; c.mvpy = mvp.y; c.lambda = lambda; c.n_int = 0; c.n_sub = 0;
    for (int k = 0; k < 5; k++) c.cyc[k] = 0;
    MeTeam<1> tm;
    tm.xch = nullptr; tm.warp = 0; tm.phase = 0;
    int mx, my;
    uint32_t cost;
    warp_motion_estimate<S, 1>(org, os, ref, rs, c, mvc.x, mvc.y, (const int16_t *)cand, ncand, mx, my, cost, tm);
    mx = __shfl_sync(FULL, mx, 0); my = __shfl_sync(FULL, my, 0); cost = __shfl_sync(FULL, cost, 0);
    mv->x = (int16_t)mx; mv->y = (int16_t)my;
    if (lane() == 0) {
      sh->prof[ST_ME] += 1; sh->prof[ST_ME_INT] += c.n_int; sh->prof[ST_ME_SUB] += c.n_sub;
      if (size <= 16)
        for (int k = 0; k < 5; k++) sh->prof[ST_MESTAGE + k] += c.cyc[k];
      sh->prof[ST_ME_SAMPLES] += (long long)(c.n_int + 1) * w * h + (long long)c.n_sub * ((w + 5) * (h + 5) + w * h);
    }
    sync();
    return (int)cost;
  }
  __device__ __noinline__ int me_bi(const S *org, int os, const S *ref0, const S *ref1, int rs, int size, Mv *mv, Mv mvc, Mv mvp, double lambda, int sign, int xpos, int ypos, const Mv *cand,
                       int ncand, S *scratch0, S *scratch1) const {
    PROF(PF_MEBI);
    sync();
    int mx, my;
    uint32_t cost;
    warp_motion_estimate_bi<S>(org, os, ref0, ref1, rs, size, sign, xpos, ypos, F->width, F->height, F->bitdepth, 1, lambda, mvc.x, mvc.y, mvp.x, mvp.y, (const int16_t *)cand,
                               ncand, mx, my, cost, scratch0, scratch1);
    mx = __shfl_sync(FULL, mx, 0); my = __shfl_sync(FULL, my, 0); cost = __shfl_sync(FULL, cost, 0);
    mv->x = (int16_t)mx; mv->y = (int16_t)my;
    sync();
    return (int)cost;
  }
  // check_early_skip_sub_block (enc/encode_block.c:2147-2180): 2x2 average of the residual, (size/2)-point transform, any |c| > threshold
  __device__ __noinline__ int es_luma(const S *orig, int os, const S *pred, int ps, int size, int threshold) const {
    PROF(PF_ES);
    const int s2 = size / 2, l2 = ilog2(s2);
    sync();
    TB_ROLL
    for (int p = lane(); p < s2 * s2; p += 32) {
      const int i = p >> l2, j = p & (s2 - 1);
      int sum = 2;
#pragma unroll
      for (int m = 0; m < 2; m++)
#pragma unroll
        for (int n = 0; n < 2; n++) sum += (int)(int16_t)((int)orig[(2 * i + m) * os + 2 * j + n] - (int)pred[(2 * i + m) * ps + 2 * j + n]);
      sh->blk16[p] = (int16_t)(sum >> 2);
    }
    sync();
    warp_fwd_transform(sh->blk16, s2, s2, 0, F->bitdepth, sh->sc, sh->out16, cta->tab16);
    int hit = 0;
    TB_ROLL
    for (int p = lane(); p < s2 * s2; p += 32) hit |= iabs((int)sh->out16[p]) > threshold;
    hit = __any_sync(FULL, hit);
    sync();
    return hit;
  }
  // check_early_skip_sub_blockC :2214-2229 with calc_cbp_simd
  __device__ __noinline__ int es_chroma(const S *orig, int os, const S *pred, int ps, int size, int threshold) const {
    PROF(PF_ES);
    const int ls = ilog2(size);
    sync();
    TB_ROLL
    for (int p = lane(); p < size * size; p += 32) {
      const int i = p >> ls, j = p & (size - 1);
      sh->blk16[p] = (int16_t)((int)orig[i * os + j] - (int)pred[i * ps + j]);
    }
    sync();
    const int r = warp_calc_cbp(sh->blk16, size, threshold);
    sync();
    return r;
  }
  __device__ __noinline__ void store_blk(tb_rdo_blk_t *blk, int stride, int by, int bx, int nbw, int nbh, int div, tb_rdo_blk_t v, const Mv *mv0, const Mv *mv1) const {
    sync();
    TB_ROLL
    for (int p = lane(); p < nbw * nbh; p += 32) {
      const int m = p / nbw, n = p - m * nbw;
      const int m0 = div > 0 ? m / div : 0, n0 = div > 0 ? n / div : 0, index = 2 * m0 + n0;
      tb_rdo_blk_t w = v;
      w.mv0 = mv0[index]; w.mv1 = mv1[index];
      blk[(by + m) * stride + bx + n] = w;
    }
    sync();
  }
  __device__ __noinline__ void pack_coeff(int16_t *dst, const int16_t *q, int size, int tb_split, int nonzero) const {
    const int t = tb_split ? size / 2 : size, qs = t < 16 ? t : 16, n = tb_split ? 4 : 1, nq = qs * qs;
    sync();
    TB_ROLL
    for (int p = lane(); p < n * nq; p += 32) {
      const int k = p / nq, i = p - k * nq;
      dst[p] = nonzero ? q[k * 256 + i] : (int16_t)0;
    }
    sync();
  }
  __device__ void store_leaf(tb_rdo_leaf_t *p, const tb_rdo_leaf_t &L) const {
    if (lane() == 0) *p = L;
    sync();
  }
  __device__ void store_count(int *p, int n) const {
    if (lane() == 0) *p = n;
    sync();
  }
};

constexpr int RDO_WARPS = 8;        // warps per CTA: 8 x 32 threads x 255 registers = the whole register file of an SM
constexpr int RDO_CTAS_PER_SM = 1;  // two CTAs per SM (128 registers) measured slower than one (profiles/r2_ncu_rdo_summary.md)

// One row of super blocks of one frame of the batch.  Rows are the unit a CTA claims; super blocks inside a row are sequential.
struct RowDesc { int frame, row, nsbx, pad; };
// scheduler words behind the per-row arrays
enum { CTL_REMAINING = 0, CTL_ERROR = 1, CTL_EVENT = 2 /* bumped after every finished super block */, CTL_N = 4 };

// Persistent CTAs draw READY super blocks from the rows of every frame of the batch (dataflow scheduling): row r of a frame may process
// super block c when row r-1 has published min(c+2, nsbx) super blocks (left, up-left, up, up-right neighbours: get_mv_pred / intra
// prediction / block contexts read nothing else); frames are independent of each other.  A CTA claims a ready row (lowest index first:
// the top rows of the earliest frames unblock the most work), processes super blocks while the next one is ready, then releases the row,
// so a CTA never holds an SM while it waits for a neighbour: a row migrates between CTAs at super-block boundaries (all per-super-block
// state is re-initialised by process_sb; data of other super blocks is read through L2, see TB_LDF above).
template <class S>
__global__ void __launch_bounds__(32 * RDO_WARPS, RDO_CTAS_PER_SM)
    rdo_batch_kernel(const FrameCtx<S> *ctxs, const RowDesc *rows, int nrows, Work<S> *works, int *prog, int *claimed, int *ctl, unsigned long long *prof_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RdoCta &cta = *(RdoCta *)smem_raw;
  FrameCtx<S> &fctx = *(FrameCtx<S> *)(smem_raw + ((sizeof(RdoCta) + 15) & ~(size_t)15));
  RdoShared<S> *shs = (RdoShared<S> *)(smem_raw + ((sizeof(RdoCta) + 15) & ~(size_t)15) + ((sizeof(FrameCtx<S>) + 15) & ~(size_t)15));
  const int nw = blockDim.x >> 5, wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  RdoShared<S> &sh = shs[wid];
  for (int k = lane; k < ST_END; k += 32) sh.prof[k] = 0;
  const long long t_start = clock64();
  dct_tab8_fill(cta.tab8, cta.tab8 + DCT_TAB8_SIZE);
  dct_tab_fill(cta.tab16);
  for (int t = threadIdx.x; t < 256; t += blockDim.x) ((uint8_t *)(cta.tab8 + 2 * DCT_TAB8_SIZE))[t] = (uint8_t)zigzag_index(t >> 4, t & 15, 16);
  __syncthreads();
  DevBackend<S> be;
  be.F = &fctx; be.sh = &sh; be.cta = &cta; be.nw = nw; be.wid = wid;
  volatile int *vprog = prog, *vclaimed = claimed, *vctl = ctl;
  long long idle_since = clock64();
  int cur_frame = -1;
  while (true) {
    // ---- claim a ready row
    int sel;
    {
      Prof pw(sh.prof, PF_WAIT);
      if (threadIdx.x == 0) { cta.sel = 0x7fffffff; cta.x_idx[1] = vctl[CTL_EVENT]; }  // the event count BEFORE the scan: progress made during the scan is not lost
      __syncthreads();
      int mine = 0x7fffffff;
      for (int g = threadIdx.x; g < nrows; g += blockDim.x) {
        if (vclaimed[g]) continue;
        const RowDesc rd = rows[g];
        const int p = vprog[g];
        if (p < rd.nsbx && (rd.row == 0 || vprog[g - 1] >= min(p + 2, rd.nsbx))) { mine = g; break; }
      }
      if (mine != 0x7fffffff) atomicMin(&cta.sel, mine);
      __syncthreads();
      sel = cta.sel;
      if (sel == 0x7fffffff) {  // nothing ready: finished, failed, or wait for the running super blocks
        if (threadIdx.x == 0) {
          // ONE thread polls ONE word (the event counter) at a low rate: a super block takes ~100 ms, and every CTA of the grid scanning the row
          // table in a tight loop turns its few cache lines into a hot spot of one L2 slice that slows the working CTAs down
          int f = 0;
          const int ev0 = cta.x_idx[1];
          while (true) {
            if (vctl[CTL_REMAINING] <= 0) { f = 1; break; }
            // ~30 s of SM clocks without any work for this CTA while work remains: a row stopped publishing (it faulted): do not hang the launch
            if (vctl[CTL_ERROR] != 0 || clock64() - idle_since > 60000000000ll) { vctl[CTL_ERROR] = 1; f = 1; break; }
            if (vctl[CTL_EVENT] != ev0) break;
            __nanosleep(20000);
          }
          cta.x_flag[0] = f;
        }
        __syncthreads();
        if (cta.x_flag[0]) break;
        continue;
      }
      if (threadIdx.x == 0) {
        int got = atomicCAS(&claimed[sel], 0, 1) == 0;
        if (got) {  // the row is ours: its position cannot change any more; re-evaluate readiness at that position
          const RowDesc rd = rows[sel];
          const int p = vprog[sel];
          if (!(p < rd.nsbx && (rd.row == 0 || vprog[sel - 1] >= min(p + 2, rd.nsbx)))) { atomicExch(&claimed[sel], 0); got = 0; }
          cta.x_idx[0] = p;
        }
        cta.x_flag[0] = got;
      }
      __syncthreads();
      if (!cta.x_flag[0]) continue;
    }
    __threadfence();
    const RowDesc rd = rows[sel];
    if (rd.frame != cur_frame) {  // frame parameters into shared memory
      const int *src = (const int *)(ctxs + rd.frame);
      int *dst = (int *)&fctx;
      __syncthreads();
      for (int k = threadIdx.x; k < (int)(sizeof(FrameCtx<S>) / 4); k += blockDim.x) dst[k] = src[k];
      cur_frame = rd.frame;
    }
    __syncthreads();
    int sbx = cta.x_idx[0];
    while (true) {
      Rdo<S, DevBackend<S>> R(fctx, works[blockIdx.x * nw + wid], works[blockIdx.x * nw], be);
      if (lane == 0) sh.t_mark = clock64();
      R.process_sb(sbx, rd.row);
      be.mark(tbr::PH_OTHER);
      __threadfence();  // every writing thread orders its stores before the flag
      __syncthreads();
      if (threadIdx.x == 0) {
        sh.prof[ST_SB] += 1;
        vprog[sel] = sbx + 1;
        atomicSub(&ctl[CTL_REMAINING], 1);
        const int nx = sbx + 1;
        const int cont = nx < rd.nsbx && (rd.row == 0 || vprog[sel - 1] >= min(nx + 2, rd.nsbx));
        if (!cont) { __threadfence(); atomicExch(&claimed[sel], 0); }
        __threadfence();
        atomicAdd(&ctl[CTL_EVENT], 1);
        cta.x_flag[0] = cont;
      }
      __syncthreads();
      if (!cta.x_flag[0]) break;
      __threadfence();
      sbx++;
    }
    idle_since = clock64();
  }
  if (lane == 0) {
    sh.prof[PF_TOTAL] = clock64() - t_start;
    for (int k = 0; k < ST_END; k++)
      if (sh.prof[k]) atomicAdd(&prof_out[k], (unsigned long long)sh.prof[k]);
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------------------------
char g_err[256] = {0};
#define CK(x)                                                                                     \
  do {                                                                                            \
    cudaError_t e__ = (x);                                                                        \
    if (e__ != cudaSuccess) { snprintf(g_err, sizeof(g_err), "%s: %s", #x, cudaGetErrorString(e__)); return TB_ERR_CUDA; } \
  } while (0)

// device-resident state of one frame of a batch
struct Slot {
  int w = 0, h = 0, esz = 0, sb = 0, pad = 0, nref = 0, sy = 0, sc = 0, used = 0;
  void *org[3] = {nullptr, nullptr, nullptr}, *rec[3] = {nullptr, nullptr, nullptr};
  void *ref[TB_RDO_MAX_REF][3] = {};
  tb_rdo_blk_t *blk = nullptr;
  tb_rdo_leaf_t *leaves = nullptr;
  int *leaf_count = nullptr;
  int16_t *coeffs = nullptr;
  int nsbx = 0, nsby = 0;
  void release() {
    for (int p = 0; p < 3; p++) { cudaFree(org[p]); cudaFree(rec[p]); org[p] = rec[p] = nullptr; }
    for (int r = 0; r < TB_RDO_MAX_REF; r++)
      for (int p = 0; p < 3; p++) { cudaFree(ref[r][p]); ref[r][p] = nullptr; }
    cudaFree(blk); cudaFree(leaves); cudaFree(leaf_count); cudaFree(coeffs);
    blk = nullptr; leaves = nullptr; leaf_count = nullptr; coeffs = nullptr; w = 0; nref = 0; used = 0;
  }
};
}  // namespace

struct tb_rdo_batch {
  int nslots = 0, esz = 0, grid = 0, nrows = 0, nrows_cap = 0, grid_cap = 0;
  Slot *slots = nullptr;
  void *ctx_host = nullptr, *ctx_dev = nullptr;  // FrameCtx<S>[nslots] (pinned staging, device copy)
  RowDesc *rows_host = nullptr, *rows_dev = nullptr;
  int *sched_dev = nullptr;                      // prog[nrows] | claimed[nrows] | ctl[CTL_N]
  int *ctl_host = nullptr;                       // pinned: ctl words read back after the launch
  void *works = nullptr;
  unsigned long long *prof = nullptr;
  unsigned long long stats[ST_END] = {};
  int sms = 0;
};

namespace {

template <class S> size_t smem_bytes() {
  return ((sizeof(RdoCta) + 15) & ~(size_t)15) + ((sizeof(FrameCtx<S>) + 15) & ~(size_t)15) + sizeof(RdoShared<S>) * RDO_WARPS;
}

int slot_prepare(Slot &D, const tb_rdo_frame_t *f) {
  const int w = f->width, h = f->height, sb = 1 << f->log2_sb_size, esz = f->sample_bytes;
  // device planes use the padded geometry of the caller's reference frames; a frame without references (intra) may leave it unset:
  // then the reference's own geometry (common/common_frame.c:435-452 with PADDING_Y = 160)
  const int pad = f->ref_stride[0] > 0 ? f->ref_pad : 160, padc = pad >> 1;
  const int sy = f->ref_stride[0] > 0 ? f->ref_stride[0] : ((w + 2 * pad + 15) & ~15), sc = f->ref_stride[0] > 0 ? f->ref_stride[1] : (((w >> 1) + 2 * padc + 15) & ~15);
  const size_t ref_y_bytes = (size_t)(h + 2 * pad) * sy * esz, ref_c_bytes = (size_t)((h >> 1) + 2 * padc) * sc * esz;
  if (D.w != w || D.h != h || D.esz != esz || D.sb != sb || D.pad != pad || D.sy != sy || D.sc != sc || D.nref < f->num_ref) {
    D.release();
    D.nsbx = (w + sb - 1) / sb; D.nsby = (h + sb - 1) / sb;
    const int nsb = D.nsbx * D.nsby;
    // source and reconstruction use the padded geometry of the reference frames (only their visible area is touched)
    for (int p = 0; p < 3; p++) { CK(cudaMalloc(&D.org[p], (p ? ref_c_bytes : ref_y_bytes) + 256)); CK(cudaMalloc(&D.rec[p], (p ? ref_c_bytes : ref_y_bytes) + 256)); }
    for (int r = 0; r < f->num_ref || r < 5; r++)
      for (int p = 0; p < 3; p++) CK(cudaMalloc(&D.ref[r][p], (p ? ref_c_bytes : ref_y_bytes) + 256));
    CK(cudaMalloc(&D.blk, sizeof(tb_rdo_blk_t) * (size_t)(h / 4) * (w / 4)));
    CK(cudaMalloc(&D.leaves, sizeof(tb_rdo_leaf_t) * (size_t)nsb * TB_RDO_MAX_LEAVES));
    CK(cudaMalloc(&D.leaf_count, sizeof(int) * nsb));
    CK(cudaMalloc(&D.coeffs, sizeof(int16_t) * (size_t)nsb * TB_RDO_SB_COEFFS));
    D.w = w; D.h = h; D.esz = esz; D.sb = sb; D.pad = pad; D.sy = sy; D.sc = sc; D.nref = f->num_ref > 5 ? f->num_ref : 5;
  }
  return TB_OK;
}

template <class S> void fill_ctx(FrameCtx<S> &C, const Slot &D, const tb_rdo_frame_t *f) {
  static const int8_t chroma_qp_mid[13] = {29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37};  // common/common_tables.c:67-72
  const int w = D.w, h = D.h, esz = D.esz, pad = D.pad, padc = pad >> 1, sy = D.sy, sc = D.sc;
  memset(&C, 0, sizeof(C));
  C.width = w; C.height = h; C.sb_size = D.sb; C.bitdepth = f->bitdepth; C.frame_type = f->frame_type; C.qp = f->qp;
  C.qpc = f->qp < 30 ? f->qp : (f->qp >= 43 ? f->qp - 6 : chroma_qp_mid[f->qp - 30]);
  C.num_ref = f->num_ref; C.interp_ref = f->interp_ref; C.num_intra_modes = f->num_intra_modes; C.lambda = f->lambda; C.sqrt_lambda = sqrt(f->lambda);
  C.enable_bipred = f->enable_bipred; C.enable_tb_split = f->enable_tb_split; C.enable_pb_split = f->enable_pb_split; C.speed = f->encoder_speed; C.intra_rdo = f->intra_rdo;
  C.use_block_contexts = f->use_block_contexts; C.cfl_intra = f->cfl_intra; C.cfl_inter = f->cfl_inter; C.early_skip_thr = f->early_skip_thr;
  const size_t oy = ((size_t)pad * sy + pad) * esz, oc = ((size_t)padc * sc + padc) * esz;
  for (int r = 0; r < TB_RDO_MAX_REF; r++) {
    C.ref_sign[r] = f->ref_sign[r]; C.ref_sign_ge[r] = f->ref_sign_ge[r];
    for (int p = 0; p < 3; p++) C.ref[r][p] = r < f->num_ref ? (const S *)((char *)D.ref[r][p] + (p ? oc : oy)) : nullptr;
  }
  for (int p = 0; p < 3; p++) { C.org[p] = (const S *)((char *)D.org[p] + (p ? oc : oy)); C.rec[p] = (S *)((char *)D.rec[p] + (p ? oc : oy)); }
  C.org_stride[0] = sy; C.org_stride[1] = sc; C.ref_stride[0] = sy; C.ref_stride[1] = sc; C.rec_stride[0] = sy; C.rec_stride[1] = sc;
  C.blk = D.blk; C.blk_stride = w / 4; C.leaves = D.leaves; C.leaf_count = D.leaf_count; C.coeffs = D.coeffs;
}

int check_desc(const tb_rdo_frame_t *f) {
  if (!f || f->num_ref > TB_RDO_MAX_REF || f->num_ref < 0 || f->log2_sb_size > 7 || f->log2_sb_size < 4 || (f->sample_bytes != 1 && f->sample_bytes != 2) || f->width <= 0 ||
      f->height <= 0 || (f->width & 7) || (f->height & 7) || f->interp_ref == 2 || f->qp < 0 || f->qp > 51 ||
      (f->num_ref > 0 && (f->ref_pad < 160 /* clip_mv admits vectors 144 samples outside the frame (+ filter taps): the reference's PADDING_Y */ ||
                          f->ref_stride[0] < f->width + 2 * f->ref_pad))) {
    snprintf(g_err, sizeof(g_err), "unsupported frame description (%dx%d, %d refs, sb %d, interp_ref %d, qp %d, pad %d)", f ? f->width : 0, f ? f->height : 0,
             f ? f->num_ref : 0, f ? f->log2_sb_size : 0, f ? f->interp_ref : 0, f ? f->qp : 0, f ? f->ref_pad : 0);
    return TB_ERR_ARG;
  }
  return TB_OK;
}

template <class S> int batch_launch(tb_rdo_batch *b, int n_active, cudaStream_t st) {
  // rows of the active slots, frame-major: the lowest index is the most urgent row
  int nrows = 0, nsb_total = 0;
  for (int s = 0; s < n_active; s++) { nrows += b->slots[s].nsby; nsb_total += b->slots[s].nsby * b->slots[s].nsbx; }
  if (nrows > b->nrows_cap) {
    cudaFreeHost(b->rows_host); cudaFree(b->rows_dev); cudaFree(b->sched_dev);
    b->rows_host = nullptr; b->rows_dev = nullptr; b->sched_dev = nullptr; b->nrows_cap = 0;
    CK(cudaMallocHost((void **)&b->rows_host, sizeof(RowDesc) * nrows));
    CK(cudaMalloc((void **)&b->rows_dev, sizeof(RowDesc) * nrows));
    CK(cudaMalloc((void **)&b->sched_dev, sizeof(int) * (2 * (size_t)nrows + CTL_N)));
    b->nrows_cap = nrows;
  }
  if (!b->ctl_host) CK(cudaMallocHost((void **)&b->ctl_host, sizeof(int) * CTL_N));
  int g = 0;
  for (int s = 0; s < n_active; s++)
    for (int r = 0; r < b->slots[s].nsby; r++) { b->rows_host[g].frame = s; b->rows_host[g].row = r; b->rows_host[g].nsbx = b->slots[s].nsbx; b->rows_host[g].pad = 0; g++; }
  b->nrows = nrows;
  const size_t smem = smem_bytes<S>();
  static bool attr_set[3] = {false, false, false};
  static int per_sm[3] = {0, 0, 0};
  if (!attr_set[sizeof(S)]) {
    CK(cudaFuncSetAttribute(rdo_batch_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[sizeof(S)], rdo_batch_kernel<S>, 32 * RDO_WARPS, smem));
    attr_set[sizeof(S)] = true;
  }
  if (!b->sms) { int dev = 0; CK(cudaGetDevice(&dev)); CK(cudaDeviceGetAttribute(&b->sms, cudaDevAttrMultiProcessorCount, dev)); }
  // persistent grid: every CTA is resident (a CTA may spin until a neighbour publishes), never more CTAs than rows
  int grid = b->sms * (per_sm[sizeof(S)] > 0 ? per_sm[sizeof(S)] : 1);
  if (grid > nrows) grid = nrows;
  if (grid > b->grid_cap) {
    cudaFree(b->works); b->works = nullptr; b->grid_cap = 0;
    CK(cudaMalloc(&b->works, sizeof(Work<S>) * (size_t)grid * RDO_WARPS));
    b->grid_cap = grid;
  }
  b->grid = grid;
  if (!b->prof) CK(cudaMalloc((void **)&b->prof, sizeof(unsigned long long) * ST_END));
  CK(cudaMemcpyAsync(b->rows_dev, b->rows_host, sizeof(RowDesc) * nrows, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(b->ctx_dev, b->ctx_host, sizeof(FrameCtx<S>) * n_active, cudaMemcpyDefault, st));
  CK(cudaMemsetAsync(b->sched_dev, 0, sizeof(int) * (2 * (size_t)nrows + CTL_N), st));
  b->ctl_host[CTL_REMAINING] = nsb_total; b->ctl_host[CTL_ERROR] = 0; b->ctl_host[2] = b->ctl_host[3] = 0;
  CK(cudaMemcpyAsync(b->sched_dev + 2 * (size_t)nrows, b->ctl_host, sizeof(int) * CTL_N, cudaMemcpyDefault, st));
  CK(cudaMemsetAsync(b->prof, 0, sizeof(unsigned long long) * ST_END, st));
  rdo_batch_kernel<S><<<grid, 32 * RDO_WARPS, smem, st>>>((const FrameCtx<S> *)b->ctx_dev, b->rows_dev, nrows, (Work<S> *)b->works, b->sched_dev, b->sched_dev + nrows,
                                                         b->sched_dev + 2 * (size_t)nrows, b->prof);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(b->ctl_host, b->sched_dev + 2 * (size_t)nrows, sizeof(int) * CTL_N, cudaMemcpyDefault, st));
  return TB_OK;
}

}  // namespace

extern "C" {
const char *tb_rdo_last_error(void) { return g_err; }
static uint64_t g_rdo_launches = 0;
uint64_t tb_rdo_launch_count(void) { return g_rdo_launches; }

tb_rdo_batch_t *tb_rdo_batch_create(int n_slots, int sample_bytes) {
  if (n_slots <= 0 || (sample_bytes != 1 && sample_bytes != 2)) { snprintf(g_err, sizeof(g_err), "tb_rdo_batch_create: bad arguments"); return nullptr; }
  if (tb_init(-1) != TB_OK) { snprintf(g_err, sizeof(g_err), "no CUDA device: %s", tb_last_error()); return nullptr; }  // no CPU path
  tb_rdo_batch *b = new tb_rdo_batch();
  b->nslots = n_slots; b->esz = sample_bytes;
  b->slots = new Slot[n_slots];
  const size_t cb = (sample_bytes == 1 ? sizeof(FrameCtx<uint8_t>) : sizeof(FrameCtx<uint16_t>)) * (size_t)n_slots;
  if (cudaMallocHost(&b->ctx_host, cb) != cudaSuccess || cudaMalloc(&b->ctx_dev, cb) != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "tb_rdo_batch_create: out of memory");
    tb_rdo_batch_destroy(b);
    return nullptr;
  }
  return b;
}

void tb_rdo_batch_destroy(tb_rdo_batch_t *b) {
  if (!b) return;
  cudaDeviceSynchronize();
  for (int s = 0; s < b->nslots; s++) b->slots[s].release();
  delete[] b->slots;
  cudaFreeHost(b->ctx_host); cudaFree(b->ctx_dev); cudaFreeHost(b->rows_host); cudaFree(b->rows_dev); cudaFree(b->sched_dev); cudaFreeHost(b->ctl_host);
  cudaFree(b->works); cudaFree(b->prof);
  delete b;
}

int tb_rdo_batch_upload(tb_rdo_batch_t *b, int slot, const tb_rdo_frame_t *f) {
  if (!b || slot < 0 || slot >= b->nslots) { snprintf(g_err, sizeof(g_err), "tb_rdo_batch_upload: bad slot"); return TB_ERR_ARG; }
  if (check_desc(f) != TB_OK) return TB_ERR_ARG;
  if (f->sample_bytes != b->esz) { snprintf(g_err, sizeof(g_err), "tb_rdo_batch_upload: sample size differs from the batch's"); return TB_ERR_ARG; }
  cudaStream_t st = (cudaStream_t)tb_stream();
  Slot &D = b->slots[slot];
  if (slot_prepare(D, f) != TB_OK) return TB_ERR_CUDA;
  const int esz = D.esz, w = D.w, h = D.h, padc = D.pad >> 1;
  const size_t oy = ((size_t)D.pad * D.sy + D.pad) * esz, oc = ((size_t)padc * D.sc + padc) * esz;
  const size_t ref_y_bytes = (size_t)(h + 2 * D.pad) * D.sy * esz, ref_c_bytes = (size_t)((h >> 1) + 2 * padc) * D.sc * esz;
  if (esz == 1) fill_ctx(((FrameCtx<uint8_t> *)b->ctx_host)[slot], D, f);
  else fill_ctx(((FrameCtx<uint16_t> *)b->ctx_host)[slot], D, f);
  // uploads: source (visible area), references (whole padded planes: one contiguous copy each)
  for (int p = 0; p < 3; p++)
    CK(cudaMemcpy2DAsync((char *)D.org[p] + (p ? oc : oy), (size_t)(p ? D.sc : D.sy) * esz, f->orig[p], (size_t)f->orig_stride[p ? 1 : 0] * esz, (size_t)(p ? w >> 1 : w) * esz,
                         p ? h >> 1 : h, cudaMemcpyDefault, st));
  for (int r = 0; r < f->num_ref; r++)
    for (int p = 0; p < 3; p++)
      CK(cudaMemcpyAsync(D.ref[r][p], (const char *)f->ref[r][p] - (p ? oc : oy), p ? ref_c_bytes : ref_y_bytes, cudaMemcpyDefault, st));
  D.used = 1;
  return TB_OK;
}

int tb_rdo_batch_run(tb_rdo_batch_t *b, int n_active) {
  if (!b || n_active <= 0 || n_active > b->nslots) { snprintf(g_err, sizeof(g_err), "tb_rdo_batch_run: bad frame count"); return TB_ERR_ARG; }
  for (int s = 0; s < n_active; s++)
    if (!b->slots[s].used) { snprintf(g_err, sizeof(g_err), "tb_rdo_batch_run: slot %d was never uploaded", s); return TB_ERR_ARG; }
  cudaStream_t st = (cudaStream_t)tb_stream();
  g_rdo_launches++;
  return b->esz == 1 ? batch_launch<uint8_t>(b, n_active, st) : batch_launch<uint16_t>(b, n_active, st);
}

int tb_rdo_batch_download(tb_rdo_batch_t *b, int slot, const tb_rdo_frame_t *f) {
  if (!b || slot < 0 || slot >= b->nslots || !b->slots[slot].used || !f || !f->blk || !f->leaves || !f->leaf_count || !f->coeffs) {
    snprintf(g_err, sizeof(g_err), "tb_rdo_batch_download: bad arguments");
    return TB_ERR_ARG;
  }
  cudaStream_t st = (cudaStream_t)tb_stream();
  const Slot &D = b->slots[slot];
  const int esz = D.esz, w = D.w, h = D.h, padc = D.pad >> 1, nsb = D.nsbx * D.nsby;
  if (f->width != w || f->height != h || f->sample_bytes != esz) { snprintf(g_err, sizeof(g_err), "tb_rdo_batch_download: geometry differs from the uploaded frame"); return TB_ERR_ARG; }
  const size_t oy = ((size_t)D.pad * D.sy + D.pad) * esz, oc = ((size_t)padc * D.sc + padc) * esz;
  for (int p = 0; p < 3; p++)
    if (f->rec[p])
      CK(cudaMemcpy2DAsync(f->rec[p], (size_t)f->rec_stride[p ? 1 : 0] * esz, (const char *)D.rec[p] + (p ? oc : oy), (size_t)(p ? D.sc : D.sy) * esz, (size_t)(p ? w >> 1 : w) * esz,
                           p ? h >> 1 : h, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(f->blk, D.blk, sizeof(tb_rdo_blk_t) * (size_t)(h / 4) * (w / 4), cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(f->leaves, D.leaves, sizeof(tb_rdo_leaf_t) * (size_t)nsb * TB_RDO_MAX_LEAVES, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(f->leaf_count, D.leaf_count, sizeof(int) * nsb, cudaMemcpyDefault, st));
  CK(cudaMemcpyAsync(f->coeffs, D.coeffs, sizeof(int16_t) * (size_t)nsb * TB_RDO_SB_COEFFS, cudaMemcpyDefault, st));
  return TB_OK;
}

int tb_rdo_batch_sync(tb_rdo_batch_t *b) {
  if (!b) return TB_ERR_ARG;
  cudaStream_t st = (cudaStream_t)tb_stream();
  CK(cudaStreamSynchronize(st));
  if (b->prof) CK(cudaMemcpy(b->stats, b->prof, sizeof(b->stats), cudaMemcpyDeviceToHost));
  if (getenv("TB_RDO_PROF") && b->prof) {
    const unsigned long long *pr = b->stats;
    static const char *names[PF_N] = {"interp", "me", "me_bi", "tx_chain", "coeff_bits", "ssd_sad", "intra", "copy_avg", "early_skip", "idle", "total"};
    fprintf(stderr, "[tb_rdo prof] %d rows on %d CTAs x %d warps:", b->nrows, b->grid, RDO_WARPS);
    for (int k = 0; k < PF_N; k++) fprintf(stderr, " %s %.1f%%", names[k], 100.0 * (double)pr[k] / (double)(pr[PF_TOTAL] ? pr[PF_TOTAL] : 1));
    {
      static const char *ph[tbr::PH_N] = {"other", "early_skip", "skip_merge_cand", "search", "inter_cand", "bipred", "intra_search", "intra_cand", "commit"};
      unsigned long long tot = 0;
      for (int k = 0; k < tbr::PH_N; k++) tot += pr[ST_PH + k];
      fprintf(stderr, "\n[tb_rdo prof] wall time of a super block by decision phase (warp 0):");
      for (int k = 0; k < tbr::PH_N; k++) fprintf(stderr, " %s %.1f%%", ph[k], 100.0 * (double)pr[ST_PH + k] / (double)(tot ? tot : 1));
    }
    {
      static const char *stg[5] = {"telescope", "candidates", "hexagon", "half-pel", "quarter-pel"};
      unsigned long long tot = 0;
      for (int k = 0; k < 5; k++) tot += pr[ST_MESTAGE + k];
      fprintf(stderr, "\n[tb_rdo prof] search stages (coding blocks <= 16):");
      for (int k = 0; k < 5; k++) fprintf(stderr, " %s %.1f%%", stg[k], 100.0 * (double)pr[ST_MESTAGE + k] / (double)(tot ? tot : 1));
    }
    fprintf(stderr, "\n[tb_rdo prof] search phase: warp 0 own searches %.0f, (intra items %.0f), barrier wait %.0f | last warp (searches %.0f) intra items %.0f, barrier wait %.0f  [Mcycles]",
            pr[ST_X] / 1e6, pr[ST_X + 1] / 1e6, pr[ST_X + 2] / 1e6, pr[ST_X + 3] / 1e6, pr[ST_X + 4] / 1e6, pr[ST_X + 5] / 1e6);
    fprintf(stderr, "\n[tb_rdo prof] search cycles by coding-block size 8..128:");
    for (int k = 0; k < 5; k++) fprintf(stderr, " %.1f%%", 100.0 * (double)pr[ST_ME_SZ + k] / (double)(pr[PF_ME] ? pr[PF_ME] : 1));
    fprintf(stderr, "; transform chains by size 4..128:");
    for (int k = 0; k < 6; k++) fprintf(stderr, " %.1f%%", 100.0 * (double)pr[ST_TX_SZ + k] / (double)(pr[PF_TX] ? pr[PF_TX] : 1));
    fprintf(stderr, "; predictions by size 4..128:");
    for (int k = 0; k < 6; k++) fprintf(stderr, " %.1f%%", 100.0 * (double)pr[ST_IP_SZ + k] / (double)(pr[PF_INTERP] ? pr[PF_INTERP] : 1));
    fprintf(stderr, "\n");
  }
  if (b->ctl_host && (b->ctl_host[CTL_ERROR] || b->ctl_host[CTL_REMAINING] != 0)) {
    snprintf(g_err, sizeof(g_err), "rdo_batch_kernel: a super-block row stopped publishing progress (%d super blocks left)", b->ctl_host[CTL_REMAINING]);
    return TB_ERR_CUDA;
  }
  return TB_OK;
}

int tb_rdo_batch_grid(const tb_rdo_batch_t *b) { return b ? b->grid : 0; }
int tb_rdo_batch_stats(const tb_rdo_batch_t *b, uint64_t *out, int n) {
  if (!b || !out) return 0;
  const int m = n < TB_RDO_NSTATS ? n : TB_RDO_NSTATS;
  for (int k = 0; k < m; k++) out[k] = b->stats[k];
  return m;
}

int tb_rdo_encode_frames(const tb_rdo_frame_t *f, int n) {
  static tb_rdo_batch *B[3] = {nullptr, nullptr, nullptr};  // one internal batch per sample size, grown on demand
  if (!f || n <= 0) { snprintf(g_err, sizeof(g_err), "tb_rdo_encode_frames: bad arguments"); return TB_ERR_ARG; }
  for (int i = 0; i < n; i++) {
    if (check_desc(&f[i]) != TB_OK) return TB_ERR_ARG;
    if (f[i].sample_bytes != f[0].sample_bytes) { snprintf(g_err, sizeof(g_err), "tb_rdo_encode_frames: mixed sample sizes"); return TB_ERR_ARG; }
    if (!f[i].blk || !f[i].leaves || !f[i].leaf_count || !f[i].coeffs) { snprintf(g_err, sizeof(g_err), "tb_rdo_encode_frames: missing output buffers"); return TB_ERR_ARG; }
  }
  const int esz = f[0].sample_bytes;
  if (!B[esz] || B[esz]->nslots < n) {
    tb_rdo_batch_destroy(B[esz]);
    B[esz] = tb_rdo_batch_create(n, esz);
    if (!B[esz]) return TB_ERR_CUDA;
  }
  int rc;
  for (int i = 0; i < n; i++)
    if ((rc = tb_rdo_batch_upload(B[esz], i, &f[i])) != TB_OK) return rc;
  if ((rc = tb_rdo_batch_run(B[esz], n)) != TB_OK) return rc;
  for (int i = 0; i < n; i++)
    if ((rc = tb_rdo_batch_download(B[esz], i, &f[i])) != TB_OK) return rc;
  return tb_rdo_batch_sync(B[esz]);
}

int tb_rdo_encode_frame(const tb_rdo_frame_t *f) { return tb_rdo_encode_frames(f, 1); }
}
