// tb_device.cuh — warp-level device routines of the Thor hot path for sm_100a.
//
// Execution model: ONE WARP PER WORK ITEM (coding / prediction / transform block, or one motion search).  Small
// blocks are packed several-probes-per-warp inside the routines so all 32 lanes stay busy.  Samples are handled as
// 32-bit words (4 x u8 or 2 x u16): VABSDIFF4.U8.ACC does the byte SAD, unaligned reference words are assembled
// from two aligned loads with a funnel shift.  Integer arithmetic follows the reference bit for bit; the only
// floating-point expression on the path (lambda * bits + 0.5, enc/encode_block.c:550) is evaluated with explicit
// round-to-nearest double mul/add so it cannot be contracted into an FMA.
//
// Every routine cites the reference function whose results it reproduces (paths relative to /root/reference).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

// TB_LDG: read-only-path load of data that no thread writes during the kernel (frames, work items).  TB_LDF: load of reconstructed
// samples that ANOTHER CTA may have written earlier in the same kernel (wavefront RD loop, tb_rdo.cu): that translation unit maps
// TB_LDG to a plain load (its "original" block can be a scratch block written moments ago) and TB_LDF to an L1-bypassing load.
#ifndef TB_SAD_ROWS
#define TB_SAD_ROWS 0
#endif
#ifndef TB_ROLL
#define TB_ROLL  // tb_rdo.cu: "#pragma unroll 1" on the simple per-sample loops (its kernel is bound by instruction fetch)
#endif
#ifndef TB_ME_STAGE_PROF
#define TB_ME_STAGE_PROF 0
#endif
#ifndef TB_LDG
#define TB_LDG(p) __ldg(p)
#endif
#ifndef TB_LDF
#define TB_LDF(p) (*(p))
#endif

namespace tb {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int ilog2(int x) { return 31 - __clz(x); }                       // common/simd.h:86
__device__ __forceinline__ int iabs(int x) { return x < 0 ? -x : x; }
__device__ __forceinline__ int iclip(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
__device__ __forceinline__ int sat_px(int v, int maxv) { return v < 0 ? 0 : (v > maxv ? maxv : v); }  // common/global.h:128

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) { return __reduce_add_sync(FULL, v); }
__device__ __forceinline__ uint64_t warp_sum64(uint64_t v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
// sum over aligned groups of `g` lanes (g power of two <= 32); every lane of a group gets the group's sum
__device__ __forceinline__ uint32_t group_sum(uint32_t v, int g) {
  for (int o = g >> 1; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------------------------
// 32-bit word access to sample rows.  PW = samples per word.
// ---------------------------------------------------------------------------------------------------------------
template <class S> struct Word { static constexpr int PW = 4 / (int)sizeof(S); };

// 32-bit load from a pointer with only sample alignment: two aligned loads + funnel shift (SHF.R.W).
__device__ __forceinline__ uint32_t ldw_any(const void *p) {
  uintptr_t a = (uintptr_t)p;
  const uint32_t *q = (const uint32_t *)(a & ~(uintptr_t)3);
  unsigned sh = (unsigned)(a & 3) * 8;
  uint32_t lo = q[0];
  if (sh == 0) return lo;
  return __funnelshift_r(lo, q[1], sh);
}
template <class S> __device__ __forceinline__ uint32_t word_sad(uint32_t a, uint32_t b) {
  return sizeof(S) == 1 ? __vsadu4(a, b) : __vsadu2(a, b);
}
template <class S> __device__ __forceinline__ int word_px(uint32_t w, int i) {
  return sizeof(S) == 1 ? (int)((w >> (8 * i)) & 0xff) : (int)((w >> (16 * i)) & 0xffff);
}

// ---------------------------------------------------------------------------------------------------------------
// a1: SAD of a w x h block.  enc/encode_block.c:417-428 / enc/enc_kernels.c:36-81.
// `o` must be 4-byte aligned with an even word pitch (original blocks always are); `r` arbitrary.
// Lanes sub..sub+nl-1 of a group share the block; returns this lane's partial sum.
// ---------------------------------------------------------------------------------------------------------------
// Rows of >= 16 bytes with 128-bit loads: one aligned LDG.128 per 16 reference bytes (+1 per row) and one per 16 original
// bytes instead of eight 32-bit loads — the search is bound by L1 wavefronts (59 % of the l1tex data-pipe peak in ncu), so
// request count matters more than bytes.  J = word offset of the row inside its first 16-byte chunk (uniform per lane group:
// all pitches are multiples of 16 bytes), sh = remaining byte offset in bits.
template <class S, int J>
__device__ __forceinline__ uint32_t sad_rows_v4(const uint4 *rq, int rsv, const uint4 *oq, int osv, int nch, int h, int sub, int nl, unsigned sh) {
  uint32_t acc = 0;
  for (int row = sub; row < h; row += nl) {
    const uint4 *q = rq + row * rsv, *a = oq + row * osv;
    uint4 P = TB_LDG(q);
    for (int c = 0; c < nch; c++) {
      const uint4 N = TB_LDG(q + c + 1), A = TB_LDG(a + c);
      const uint32_t w0 = J == 0 ? P.x : (J == 1 ? P.y : (J == 2 ? P.z : P.w)), w1 = J == 0 ? P.y : (J == 1 ? P.z : (J == 2 ? P.w : N.x)),
                     w2 = J == 0 ? P.z : (J == 1 ? P.w : (J == 2 ? N.x : N.y)), w3 = J == 0 ? P.w : (J == 1 ? N.x : (J == 2 ? N.y : N.z)),
                     w4 = J == 0 ? N.x : (J == 1 ? N.y : (J == 2 ? N.z : N.w));
      acc += word_sad<S>(A.x, __funnelshift_r(w0, w1, sh)) + word_sad<S>(A.y, __funnelshift_r(w1, w2, sh)) + word_sad<S>(A.z, __funnelshift_r(w2, w3, sh)) +
             word_sad<S>(A.w, __funnelshift_r(w3, w4, sh));
      P = N;
    }
  }
  return acc;
}

template <class S, bool V4 = false>
__device__ __forceinline__ uint32_t sad_partial(const S *o, int os, const S *r, int rs, int w, int h, int sub, int nl) {
  // Lane `sub` of `nl` takes the rows sub, sub+nl, ... (nl <= h).  Row pitches are multiples of 4 bytes, so the byte
  // misalignment of the reference row is the same for every row: one aligned word stream per row, one funnel shift per word.
  constexpr int PW = Word<S>::PW;
  const int ww = w / PW;  // words per row: 1, 2, 4, 8, 16, 32 (64 for 128-wide u16)
  const uintptr_t ra = (uintptr_t)r;
  const unsigned sh = (unsigned)(ra & 3) * 8;
  const uint32_t *rq = (const uint32_t *)(ra & ~(uintptr_t)3);
  const uint32_t *oq = (const uint32_t *)o;
  const int rsw = (rs * (int)sizeof(S)) >> 2, osw = (os * (int)sizeof(S)) >> 2;  // pitches in words
  if (V4 && !(ww & 3) && !((((uintptr_t)o) | (unsigned)(osw << 2) | (unsigned)(rsw << 2)) & 15)) {
    const uint4 *rv = (const uint4 *)(ra & ~(uintptr_t)15), *ov = (const uint4 *)o;
    const unsigned sh8 = (unsigned)(ra & 3) * 8;
    switch ((unsigned)(ra >> 2) & 3) {
      case 0: return sad_rows_v4<S, 0>(rv, rsw >> 2, ov, osw >> 2, ww >> 2, h, sub, nl, sh8);
      case 1: return sad_rows_v4<S, 1>(rv, rsw >> 2, ov, osw >> 2, ww >> 2, h, sub, nl, sh8);
      case 2: return sad_rows_v4<S, 2>(rv, rsw >> 2, ov, osw >> 2, ww >> 2, h, sub, nl, sh8);
      default: return sad_rows_v4<S, 3>(rv, rsw >> 2, ov, osw >> 2, ww >> 2, h, sub, nl, sh8);
    }
  }
  uint32_t acc = 0;
  TB_ROLL
  for (int row = sub; row < h; row += nl) {
    const uint32_t *q = rq + row * rsw, *a = oq + row * osw;
    uint32_t prev = TB_LDG(q);
    TB_ROLL
    for (int c = 0; c < ww; c++) {
      uint32_t nxt = TB_LDG(q + c + 1);
      acc += word_sad<S>(TB_LDG(a + c), __funnelshift_r(prev, nxt, sh));
      prev = nxt;
    }
  }
  return acc;
}
// whole warp on one block
template <class S> __device__ __forceinline__ uint32_t warp_sad(const S *o, int os, const S *r, int rs, int w, int h) {
  return warp_sum(lane_id() < h ? sad_partial<S>(o, os, r, rs, w, h, lane_id(), 32) : 0u);
}

// SADs of up to 32 reference positions of the same block: lane i supplies the sample offset `roff` of position i
// (i < n); lane i receives SAD i.  L = lanes cooperating on one position = words/16 (1 for blocks up to 8x8 u8: the
// whole 5x5 telescope grid is then evaluated in ONE pass, one position per lane, no shuffles), 32 for >= 512 words.
template <class S>
__device__ __noinline__ uint32_t multi_sad_narrow(const S *o, int os, const S *r, int rs, int w, int h, int roff, int n) {
  constexpr int PW = Word<S>::PW;
  const int lane = lane_id();
  const int nwords = (w / PW) * h;
  int L = nwords >= 512 ? 32 : (nwords <= 16 ? 1 : nwords >> 4);  // power of two
  if (L > h) L = h;  // rows are dealt to lanes
  // few positions (hexagon rounds: 3-6, candidate lists): widen the lane group per position while everything still fits one pass
  while (L < 32 && 2 * L * n <= 32 && 2 * L <= h) L *= 2;
  uint32_t out = 0;
  if (L == 32) {
    for (int p = 0; p < n; p++) {
      int off = __shfl_sync(FULL, roff, p);
      uint32_t s = warp_sum(lane < h ? sad_partial<S>(o, os, r + off, rs, w, h, lane, 32) : 0u);
      if (lane == p) out = s;
    }
  } else if (L == 1) {
    if (lane < n) out = sad_partial<S>(o, os, r + roff, rs, w, h, 0, 1);
  } else {
    const int g = 32 / L;  // positions per pass
    const int sub = lane & (L - 1), grp = lane / L;
    for (int base = 0; base < n; base += g) {
      int p = base + grp;
      int off = __shfl_sync(FULL, roff, p & 31);
      uint32_t s = (p < n) ? sad_partial<S>(o, os, r + off, rs, w, h, sub, L) : 0u;
      s = group_sum(s, L);
      uint32_t got = __shfl_sync(FULL, s, ((lane - base) * L) & 31);
      if (lane >= base && lane < base + g && lane < n) out = got;
    }
  }
  return out;
}

// The same for blocks of >= 256 words whose rows are >= 16 bytes: 16 or 32 lanes per position, so at most two positions (two
// chunk offsets) are in flight per pass and the 128-bit row loads of sad_rows_v4 stay (nearly) uniform.  A separate function:
// its larger register footprint must not be paid around the calls for small blocks.
template <class S>
__device__ __noinline__ uint32_t multi_sad_wide(const S *o, int os, const S *r, int rs, int w, int h, int roff, int n) {
  constexpr int PW = Word<S>::PW;
  const int lane = lane_id();
  const int nwords = (w / PW) * h;
  int L = nwords >= 512 ? 32 : 16;
  if (L > h) L = h;  // h >= 16 here
  uint32_t out = 0;
  if (L == 32) {
    for (int p = 0; p < n; p++) {
      int off = __shfl_sync(FULL, roff, p);
      uint32_t s = warp_sum(lane < h ? sad_partial<S, true>(o, os, r + off, rs, w, h, lane, 32) : 0u);
      if (lane == p) out = s;
    }
  } else {
    const int sub = lane & 15, grp = lane >> 4;
    for (int base = 0; base < n; base += 2) {
      int p = base + grp;
      int off = __shfl_sync(FULL, roff, p & 31);
      uint32_t s = (p < n) ? sad_partial<S, true>(o, os, r + off, rs, w, h, sub, 16) : 0u;
      s = group_sum(s, 16);
      uint32_t got = __shfl_sync(FULL, s, ((lane - base) * 16) & 31);
      if (lane >= base && lane < base + 2 && lane < n) out = got;
    }
  }
  return out;
}
// The same for the device-resident RD loop (tb_rdo.cu, TB_SAD_ROWS), where ONE warp walks blocks of up to 128x128 alone and nothing else hides its latency:
// the lanes of a load request lie along a ROW (32-byte .. 128-byte contiguous segments: one or two L1 wavefronts per request instead of one per lane when
// the rows are dealt to lanes), five positions share each load of the original (a telescope grid row: their reference segments overlap), and the five
// accumulations are independent.  Rows >= 8 words; lane = (row % RP) * LW + word, RP rows per pass.
template <class S>
__device__ __noinline__ uint32_t multi_sad_rows(const S *o, int os, const S *r, int rs, int w, int h, int roff, int n) {
  constexpr int PW = Word<S>::PW, CH = 5;
  const int lane = lane_id();
  const int LW = w / PW, LWe = LW < 32 ? LW : 32, RP = 32 / LWe, CI = LW / LWe;  // words per row, lanes per row, rows per pass, column iterations
  const int col0 = lane & (LWe - 1), rsub = lane / LWe;
  const int osw = (os * (int)sizeof(S)) >> 2;
  const uint32_t *oq = (const uint32_t *)o;
  uint32_t out = 0;
  for (int base = 0; base < n; base += CH) {
    const uint32_t *rq[CH];
    unsigned sh[CH];
#pragma unroll
    for (int k = 0; k < CH; k++) {
      const int off = __shfl_sync(FULL, roff, min(base + k, n - 1));
      const uintptr_t a = (uintptr_t)(r + off);
      rq[k] = (const uint32_t *)(a & ~(uintptr_t)3);
      sh[k] = (unsigned)(a & 3) * 8;
    }
    const int rsw = (rs * (int)sizeof(S)) >> 2;
    uint32_t acc[CH] = {0, 0, 0, 0, 0};
    TB_ROLL
    for (int row = rsub; row < h; row += RP) {
      TB_ROLL
      for (int ci = 0; ci < CI; ci++) {
        const int col = col0 + ci * 32;
        const uint32_t a = TB_LDG(oq + row * osw + col);
#pragma unroll
        for (int k = 0; k < CH; k++) {
          const uint32_t *q = rq[k] + row * rsw + col;
          acc[k] += word_sad<S>(a, __funnelshift_r(TB_LDG(q), TB_LDG(q + 1), sh[k]));
        }
      }
    }
#pragma unroll
    for (int k = 0; k < CH; k++) {
      const uint32_t t = warp_sum(acc[k]);
      if (lane == base + k && base + k < n) out = t;
    }
  }
  return out;
}
template <class S, int TW = 1>
__device__ __forceinline__ uint32_t multi_sad(const S *o, int os, const S *r, int rs, int w, int h, int roff, int n) {
  // only the CTA-team searches (blocks >= 2048 samples) take the wide form: a second callee at the call sites of the one-warp
  // searches costs them more in spills than the 32x32 blocks would gain
  if (TW > 1 && (w / Word<S>::PW) * h >= 256 && h >= 16 && w * (int)sizeof(S) >= 16) return multi_sad_wide<S>(o, os, r, rs, w, h, roff, n);
#if TB_SAD_ROWS
  if (TW == 1 && w / Word<S>::PW >= 8) return multi_sad_rows<S>(o, os, r, rs, w, h, roff, n);
#endif
  return multi_sad_narrow<S>(o, os, r, rs, w, h, roff, n);
}

// a3: SSD.  enc/encode_block.c:455-465
template <class S> __device__ __forceinline__ uint64_t warp_ssd(const S *a, int as, const S *b, int bs, int w, int h) {
  uint64_t acc = 0;
  const int lw = ilog2(w);
  TB_ROLL
  for (int p = lane_id(); p < (h << lw); p += 32) {
    int row = p >> lw, col = p & (w - 1);
    int d = (int)a[row * as + col] - (int)b[row * bs + col];
    acc += (uint64_t)(uint32_t)(d * d);
  }
  return warp_sum64(acc);
}

// ---------------------------------------------------------------------------------------------------------------
// a6: MV helpers.  enc/encode_block.c:467-515, common/inter_prediction.c:51-63
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int mv_len(int d) {
  int a = iabs(d);
  if (a < 1) return 2;
  if (a < 2) return 4;
  if (a < 4) return 5;
  if (a < 36) return 5 + ((a - 4) >> 3) + 1;
  return 10 + ((a - 36) >> 4) + 1;
}
__device__ __forceinline__ int quote_mv_bits(int dy, int dx) { return mv_len(dx) + mv_len(dy); }

__device__ __forceinline__ void clip_mv(int &mvx, int &mvy, int ypos, int xpos, int fw, int fh, int bw, int bh, int sign) {
  const int ext = 160 - 16;  // PADDING_Y - 16, common/global.h:62
  int y = sign ? -mvy : mvy, x = sign ? -mvx : mvx;
  if (ypos + y / 4 < -ext) y = 4 * (-ext - ypos);
  if (ypos + y / 4 + bh > fh + ext) y = 4 * (fh + ext - ypos - bh);
  if (xpos + x / 4 < -ext) x = 4 * (-ext - xpos);
  if (xpos + x / 4 + bw > fw + ext) x = 4 * (fw + ext - xpos - bw);
  // results are stored back into int16_t mv_t fields by the reference
  mvy = (int)(int16_t)(sign ? -y : y);
  mvx = (int)(int16_t)(sign ? -x : x);
}
// lambda * bits + 0.5 in ISO-C double arithmetic (no contraction), truncated like the reference's casts
__device__ __forceinline__ uint32_t mv_cost(double lambda, int bits) {
  return (uint32_t)(int)__dadd_rn(__dmul_rn(lambda, (double)bits), 0.5);
}

// ---------------------------------------------------------------------------------------------------------------
// a7/a8: interpolation taps.  common/common_kernels.c:1905-1928
// ---------------------------------------------------------------------------------------------------------------
__constant__ int8_t c_luma_taps[2][4][6] = {
    {{0, 0, 64, 0, 0, 0}, {1, -7, 55, 19, -5, 1}, {1, -7, 38, 38, -7, 1}, {1, -5, 19, 55, -7, 1}},
    {{0, 0, 64, 0, 0, 0}, {2, -10, 59, 17, -5, 1}, {1, -8, 39, 39, -8, 1}, {1, -5, 17, 59, -10, 2}}};
__constant__ int8_t c_chroma_taps[8][4] = {{0, 64, 0, 0},  {-2, 58, 10, -2}, {-4, 54, 16, -2}, {-4, 44, 28, -4},
                                           {-4, 36, 36, -4}, {-4, 28, 44, -4}, {-2, 16, 54, -4}, {-2, 10, 58, -2}};

// One luma sample at fractional position (xf,yf) in quarter-pels; ip = integer position.
// common/inter_prediction.c:146-180.  bip = sequence-level enable_bipred value (0/1/2).
template <class S> __device__ __forceinline__ int luma_sample(const S *ip, int is, int xf, int yf, int bip, int maxv) {
  if (xf == 2 && yf == 2 && bip < 2) {
    int s = (int)ip[-is] + ip[-is + 1] + ip[-1] + ip[2] + ip[is - 1] + ip[is + 2] + ip[2 * is] + ip[2 * is + 1] +
            2 * ((int)ip[0] + ip[1] + ip[is] + ip[is + 1]);
    return sat_px((s + 8) >> 4, maxv);
  }
  const int8_t *fv = c_luma_taps[bip ? 1 : 0][yf], *fh = c_luma_taps[bip ? 1 : 0][xf];
  int sum;
  if (xf == 0) {
    sum = 0;
#pragma unroll
    for (int m = 0; m < 6; m++) sum += fv[m] * (int)ip[(m - 2) * is];
    sum *= 64;
  } else if (yf == 0) {
    sum = 0;
#pragma unroll
    for (int n = 0; n < 6; n++) sum += fh[n] * (int)ip[n - 2];
    sum *= 64;
  } else {
    sum = 0;
#pragma unroll
    for (int n = 0; n < 6; n++) {
      int col = 0;
#pragma unroll
      for (int m = 0; m < 6; m++) col += fv[m] * (int)ip[(m - 2) * is + n - 2];
      sum += fh[n] * col;
    }
  }
  return sat_px((sum + 2048) >> 12, maxv);
}
// common/inter_prediction.c:94-114
template <class S> __device__ __forceinline__ int chroma_sample(const S *ip, int is, int xf, int yf, int maxv) {
  const int8_t *fh = c_chroma_taps[xf], *fv = c_chroma_taps[yf];
  int sum = 0;
#pragma unroll
  for (int m = 0; m < 4; m++) {
    int row = 0;
#pragma unroll
    for (int n = 0; n < 4; n++) row += fh[n] * (int)ip[(m - 1) * is + n - 1];
    sum += fv[m] * row;
  }
  return sat_px((sum + 2048) >> 12, maxv);
}

// Integer part + fraction of an MV with the reference's normative clamp (lower bounds use xpos on both axes).
// common/inter_prediction.c:121-131 (luma, shift 2) and :71-81 (chroma, shift 3).
__device__ __forceinline__ void split_mv(int mvx, int mvy, int sign, int shift, int pic_w, int pic_h, int xpos, int ypos, int w, int h,
                                         int &hor_int, int &ver_int, int &xf, int &yf) {
  int x = sign ? -mvx : mvx, y = sign ? -mvy : mvy;
  int mask = (1 << shift) - 1;
  yf = y & mask;
  xf = x & mask;
  ver_int = y >> shift;
  hor_int = x >> shift;
  ver_int = min(ver_int, pic_h - ypos);
  ver_int = max(ver_int, -xpos - h);
  hor_int = min(hor_int, pic_w - xpos);
  hor_int = max(hor_int, -xpos - w);
}

__device__ void warp_interp_strips_u8(uint8_t *dst, int ds, const uint8_t *ip, int rs, int w, int h, int xf, int yf, int bip);
// Whole-warp prediction of one block into dst (common/inter_prediction.c:117-183 / :65-115).
template <class S>
__device__ void warp_interp(S *dst, int ds, const S *ref, int rs, int w, int h, int mvx, int mvy, int sign, int chroma, int bip, int pic_w,
                            int pic_h, int xpos, int ypos, int bitdepth, int sub = -1, int nl = 32) {
  // sub/nl: the block is shared by the nl lanes sub = 0 .. nl - 1 (default: the whole warp; lane groups of 8 for small blocks)
  if (sub < 0) sub = lane_id();
  int hi, vi, xf, yf;
  split_mv(mvx, mvy, sign, chroma ? 3 : 2, pic_w, pic_h, xpos, ypos, w, h, hi, vi, xf, yf);
  const S *ip = ref + vi * rs + hi;
  const int maxv = (1 << bitdepth) - 1, lw = ilog2(w);
  if (nl == 32 && sizeof(S) == 1 && !chroma && (xf | yf) && w * h >= 256 && !(h & 7) && !((((uintptr_t)dst) | (unsigned)ds | (unsigned)rs) & 3)) {
    // large 8-bit luma blocks: separable DP4A strips (same arithmetic as the search's sub-pel SAD), word stores
    warp_interp_strips_u8((uint8_t *)dst, ds, (const uint8_t *)ip, rs, w, h, xf, yf, bip);
    return;
  }
  TB_ROLL
  for (int p = sub; p < (h << lw); p += nl) {
    int row = p >> lw, col = p & (w - 1);
    const S *q = ip + row * rs + col;
    int v;
    if (xf == 0 && yf == 0) v = q[0];
    else v = chroma ? chroma_sample<S>(q, rs, xf, yf, maxv) : luma_sample<S>(q, rs, xf, yf, bip, maxv);
    dst[row * ds + col] = (S)v;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// 8-bit sub-pel SAD with DP4A: the 6x6 luma filter is separable and exact in integers, so each 4-sample-wide strip
// is filtered horizontally with two DP4A per sample (u8 samples x s8 taps), the six most recent filtered rows are kept
// in registers, and the vertical pass is 6 MADs per sample — ~12 instructions per sample instead of ~110 for the direct
// 36-tap form.  Zero fractions use the identity taps {0,0,64,0,0,0}; the (2,2) centre position uses its own 12-tap
// kernel (common/inter_prediction.c:146-158) as two row filters [0,1,1,0] / [1,2,2,1].
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_s8x4(int a, int b, int c, int d) {
  return (uint32_t)(a & 0xff) | ((uint32_t)(b & 0xff) << 8) | ((uint32_t)(c & 0xff) << 16) | ((uint32_t)(d & 0xff) << 24);
}
// u8 x s8 dot product of four byte pairs, accumulated in s32 (DP4A with mixed signedness)
__device__ __forceinline__ int dp4a_us(uint32_t a_u8x4, uint32_t b_s8x4, int c) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_s8x4), "r"(c));
  return d;
}
// four s32 -> four saturated u8 packed in one word: two I2IP (cvt.pack.sat.u8.s32)
__device__ __forceinline__ uint32_t pack_sat_u8x4(int a0, int a1, int a2, int a3) {
  // d = (sat(a) << 8) | sat(b) | (c << 16): pack the high pair first, then the low pair with the high pair as `c`
  uint32_t hi, d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(hi) : "r"(a3), "r"(a2), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a1), "r"(a0), "r"(hi));
  return d;
}
// horizontal taps on one row for the 4 outputs at p[0..3]; reads bytes p[-2..9] through aligned words
__device__ __forceinline__ void hfilt4_u8(const uint8_t *p, uint32_t tlo, uint32_t thi, int (&out)[4]) {
  uintptr_t a = (uintptr_t)(p - 2);
  const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
  const unsigned sh = (unsigned)(a & 3) * 8;
  const uint32_t w0 = TB_LDG(w), w1 = TB_LDG(w + 1), w2 = TB_LDG(w + 2), w3 = TB_LDG(w + 3);
  const uint32_t b0 = __funnelshift_r(w0, w1, sh), b1 = __funnelshift_r(w1, w2, sh), b2 = __funnelshift_r(w2, w3, sh);
#pragma unroll
  for (int k = 0; k < 4; k++) {
    uint32_t lo = __funnelshift_r(b0, b1, 8 * k), hi = __funnelshift_r(b1, b2, 8 * k);
    out[k] = dp4a_us(lo, tlo, dp4a_us(hi, thi, 0));
  }
}
// SAD of the rows [y0, y0+nrows) of one 4-wide strip at column x0 of the block; ip = integer-position sample (0,0)
// STORE = false: SAD against the original rows o; STORE = true: the prediction is written to o (a uint8_t *, 4-byte aligned rows)
template <bool STORE>
__device__ __forceinline__ uint32_t strip_subpel_u8(const uint8_t *o, int os, const uint8_t *ip, int rs, int x0, int y0, int nrows, int xf, int yf, int bip) {
  uint32_t acc = 0;
  if (xf == 2 && yf == 2 && bip < 2) {
    const uint32_t a_lo = pack_s8x4(0, 0, 1, 1), b_lo = pack_s8x4(0, 1, 2, 2), b_hi = pack_s8x4(1, 0, 0, 0);
    int h1m[4], h2a[4], h2b[4], h1p[4];  // H1[y-1], H2[y], H2[y+1], H1[y+2]
    int t1[4], t2[4];
    // prime rows y0-1, y0, y0+1
    hfilt4_u8(ip + (y0 - 1) * rs + x0, a_lo, 0, h1m);
    hfilt4_u8(ip + y0 * rs + x0, b_lo, b_hi, h2a);
    hfilt4_u8(ip + y0 * rs + x0, a_lo, 0, t1);  // H1[y0] (becomes H1[y-1] of the next row)
    hfilt4_u8(ip + (y0 + 1) * rs + x0, b_lo, b_hi, h2b);
    hfilt4_u8(ip + (y0 + 1) * rs + x0, a_lo, 0, t2);  // H1[y0+1]
    for (int y = y0; y < y0 + nrows; y++) {
      int n2[4];
      hfilt4_u8(ip + (y + 2) * rs + x0, a_lo, 0, h1p);
      hfilt4_u8(ip + (y + 2) * rs + x0, b_lo, b_hi, n2);
      uint32_t pk = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        int v = (h1m[k] + h2a[k] + h2b[k] + h1p[k] + 8) >> 4;  // max 12*255+8 -> <= 191: already inside 0..255
        pk |= (uint32_t)v << (8 * k);
      }
      if (STORE) *(uint32_t *)(const_cast<uint8_t *>(o) + y * os + x0) = pk;
      else acc += __vsadu4(TB_LDG((const uint32_t *)(o + y * os + x0)), pk);
#pragma unroll
      for (int k = 0; k < 4; k++) { h1m[k] = t1[k]; t1[k] = t2[k]; t2[k] = h1p[k]; h2a[k] = h2b[k]; h2b[k] = n2[k]; }
    }
    return acc;
  }
  const int8_t *fh = c_luma_taps[bip ? 1 : 0][xf], *fv = c_luma_taps[bip ? 1 : 0][yf];
  const uint32_t tlo = pack_s8x4(fh[0], fh[1], fh[2], fh[3]), thi = pack_s8x4(fh[4], fh[5], 0, 0);
  const int v0 = fv[0], v1 = fv[1], v2 = fv[2], v3 = fv[3], v4 = fv[4], v5 = fv[5];
  int H[6][4];  // filtered rows y-2 .. y+3
#pragma unroll
  for (int m = 0; m < 5; m++) hfilt4_u8(ip + (y0 - 2 + m) * rs + x0, tlo, thi, H[m + 1]);
  for (int y = y0; y < y0 + nrows; y++) {
#pragma unroll
    for (int m = 0; m < 5; m++)
#pragma unroll
      for (int k = 0; k < 4; k++) H[m][k] = H[m + 1][k];
    hfilt4_u8(ip + (y + 3) * rs + x0, tlo, thi, H[5]);
    int r4[4];
#pragma unroll
    for (int k = 0; k < 4; k++)
      r4[k] = (v0 * H[0][k] + v1 * H[1][k] + v2 * H[2][k] + v3 * H[3][k] + v4 * H[4][k] + v5 * H[5][k] + 2048) >> 12;
    const uint32_t pk = pack_sat_u8x4(r4[0], r4[1], r4[2], r4[3]);
    if (STORE) *(uint32_t *)(const_cast<uint8_t *>(o) + y * os + x0) = pk;
    else acc += __vsadu4(TB_LDG((const uint32_t *)(o + y * os + x0)), pk);
  }
  return acc;
}

__device__ __forceinline__ uint32_t strip_sad_subpel_u8(const uint8_t *o, int os, const uint8_t *ip, int rs, int x0, int y0, int nrows, int xf, int yf, int bip) {
  return strip_subpel_u8<false>(o, os, ip, rs, x0, y0, nrows, xf, yf, bip);
}
// prediction of a w x h luma block (w * h >= 256, h a multiple of 8): (4-column, 8-row) units dealt to the 32 lanes
__device__ __noinline__ void warp_interp_strips_u8(uint8_t *dst, int ds, const uint8_t *ip, int rs, int w, int h, int xf, int yf, int bip) {
  const int nseg = h >> 3, units = (w >> 2) * nseg;
  for (int u = lane_id(); u < units; u += 32) {
    const int strip = u / nseg, seg = u - strip * nseg;
    strip_subpel_u8<true>(dst, ds, ip, rs, strip * 4, seg * 8, 8, xf, yf, bip);
  }
}

// SADs between the original block and the luma predictions at EIGHT fractional MVs (one half-pel or quarter-pel stage of
// enc/encode_block.c:625-663) without materialising the predictions: probe t = lane / 4 uses MV (mvx0 + dx[t], mvy0 + dy[t]),
// its four lanes share the block's samples.  Every lane of probe t returns SAD t.
template <class S>
__device__ __noinline__ uint32_t subpel_stage_sads(const S *o, int os, const S *ref, int rs, int w, int hfull, int mvx, int mvy, int sign, int bip, int pic_w, int pic_h,
                                      int xpos, int ypos, int bitdepth, int row0, int h) {
  // rows [row0, row0 + h) of the w x hfull block (a team of warps splits the block into row bands; one warp: row0 = 0, h = hfull)
  int hi, vi, xf, yf;
  split_mv(mvx, mvy, sign, 2, pic_w, pic_h, xpos, ypos, w, hfull, hi, vi, xf, yf);
  const S *ip = ref + (vi + row0) * rs + hi;
  o += row0 * os;
  const int maxv = (1 << bitdepth) - 1, lw = ilog2(w), sub = lane_id() & 3;
  uint32_t acc = 0;
  if (sizeof(S) == 1) {
    // units of 4 columns x RH rows, dealt round-robin to the probe's four lanes
    // segment height: tall enough to amortise the 5-row filter halo, short enough to give every lane of the probe work
    const int RH = h >= 8 ? 8 : h, nseg = h / RH, units = (w >> 2) * nseg;
    for (int u = sub; u < units; u += 4) {
      int strip = u / nseg, seg = u - strip * nseg;
      acc += strip_sad_subpel_u8((const uint8_t *)o, os, (const uint8_t *)ip, rs, strip * 4, seg * RH, RH, xf, yf, bip);
    }
    return group_sum(acc, 4);
  }
  for (int p = sub; p < (h << lw); p += 4) {
    int row = p >> lw, col = p & (w - 1);
    const S *q = ip + row * rs + col;
    int v = (xf == 0 && yf == 0) ? (int)q[0] : luma_sample<S>(q, rs, xf, yf, bip, maxv);
    acc += (uint32_t)iabs((int)o[row * os + col] - v);
  }
  return group_sum(acc, 4);
}

// ---------------------------------------------------------------------------------------------------------------
// The half-pel stage (enc/encode_block.c:625-645) for 8-bit samples when the centre is an integer position: its eight
// probes read only THREE interpolated planes — the horizontal half-pel plane (probes (0,-2), (0,+2) in (dy,dx)), the vertical
// one ((-2,0), (+2,0)) and the 12-tap centre-kernel plane (the four diagonals) — each shifted by 0 or 1 sample.  So every plane
// sample is computed once and compared with the original at its two (four) shifts, instead of interpolating eight blocks:
// three flat passes over (plane row, 4-sample strip) units, one unit per lane and step, no state carried between units.
//   H pass: five outputs of the 6-tap row filter (two DP4A each), rounded (H + 32) >> 6 (= (64 H + 2048) >> 12), two SADs;
//   V pass: the six row words of a strip are byte-transposed with PRMT so that the column filter is two DP4A per sample;
//   C pass: H1 = [0 0 1 1 0 0] on rows r-1, r+2 and H2 = [0 1 2 2 1 0] on rows r, r+1 accumulate in one DP4A chain, four SADs.
// Lane t < 8 returns the SAD of probe t + 1; 0xffffffff = geometry not of this form (clamped vectors): use the per-probe path.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void row12_u8(const uint8_t *p, uint32_t &b0, uint32_t &b1, uint32_t &b2) {  // bytes p[0..11]
  const uintptr_t a = (uintptr_t)p;
  const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
  const unsigned sh = (unsigned)(a & 3) * 8;
  const uint32_t w0 = TB_LDG(w), w1 = TB_LDG(w + 1), w2 = TB_LDG(w + 2), w3 = TB_LDG(w + 3);
  b0 = __funnelshift_r(w0, w1, sh); b1 = __funnelshift_r(w1, w2, sh); b2 = __funnelshift_r(w2, w3, sh);
}
__device__ __noinline__ uint32_t halfpel_stage_sads_u8(const uint8_t *o, int os, const uint8_t *ref, int rs, int w, int hfull, int bx, int by, const int8_t *dxs,
                                                       const int8_t *dys, int sign, int bip, int pic_w, int pic_h, int xpos, int ypos, int row0, int h) {
  const int lane = lane_id(), t = lane & 7;
  const int mvx = (int)(int16_t)(bx + dxs[t + 1]), mvy = (int)(int16_t)(by + dys[t + 1]);
  int hi, vi, xf, yf;
  split_mv(mvx, mvy, sign, 2, pic_w, pic_h, xpos, ypos, w, hfull, hi, vi, xf, yf);
  const int hmin = __reduce_min_sync(FULL, hi), vmin = __reduce_min_sync(FULL, vi);
  const int ho = hi - hmin, vo = vi - vmin;
  const int cls = (xf == 2 && yf == 0) ? 0 : ((xf == 0 && yf == 2) ? 1 : ((xf == 2 && yf == 2) ? 2 : 3));
  const unsigned mH = __ballot_sync(FULL, cls == 0), mV = __ballot_sync(FULL, cls == 1);
  const int voH = __shfl_sync(FULL, vo, mH ? __ffs(mH) - 1 : 0), hoV = __shfl_sync(FULL, ho, mV ? __ffs(mV) - 1 : 0);
  const bool ok = bip < 2 && cls != 3 && ho <= 1 && vo <= 1 && (cls != 0 || vo == voH) && (cls != 1 || ho == hoV);
  if (!__all_sync(FULL, ok)) return 0xffffffffu;
  const int8_t *fh = c_luma_taps[bip ? 1 : 0][2];
  const uint32_t tlo = pack_s8x4(fh[0], fh[1], fh[2], fh[3]), thi = pack_s8x4(fh[4], fh[5], 0, 0);
  const int ns = w >> 2, lns = ilog2(ns);
  const uint8_t *rb = ref + (row0 + vmin) * rs + hmin;  // plane sample (r, c) <-> rb[r * rs + c]
  const uint8_t *ob = o + row0 * os;
  uint32_t aH0 = 0, aH1 = 0, aV0 = 0, aV1 = 0, aC00 = 0, aC01 = 0, aC10 = 0, aC11 = 0;  // aC<vo><ho>
  // ---- H pass: block rows y (plane rows y + voH), plane columns 4 s .. 4 s + 4
  if (mH) {
    for (int u = lane; u < h * ns; u += 32) {
      const int y = u >> lns, st = u & (ns - 1);
      uint32_t b0, b1, b2;
      row12_u8(rb + (y + voH) * rs + 4 * st - 2, b0, b1, b2);
      int v[5];
#pragma unroll
      for (int k = 0; k < 5; k++) {
        const uint32_t lo = k < 4 ? __funnelshift_r(b0, b1, 8 * k) : b1, hi4 = k < 4 ? __funnelshift_r(b1, b2, 8 * k) : b2;
        v[k] = (dp4a_us(lo, tlo, dp4a_us(hi4, thi, 32))) >> 6;
      }
      const uint32_t ow = TB_LDG((const uint32_t *)(ob + y * os + 4 * st));
      aH0 += __vsadu4(ow, pack_sat_u8x4(v[0], v[1], v[2], v[3]));
      aH1 += __vsadu4(ow, pack_sat_u8x4(v[1], v[2], v[3], v[4]));
    }
  }
  // ---- V pass: plane rows r = 0 .. h, plane columns 4 s + hoV .. + 3; row r serves block row r (vo 0) and r - 1 (vo 1)
  if (mV) {
    for (int u = lane; u < (h + 1) * ns; u += 32) {
      const int r = u >> lns, st = u & (ns - 1);
      const uint8_t *p = rb + (r - 2) * rs + 4 * st + hoV;
      const uintptr_t a = (uintptr_t)p;
      const uint32_t *wq = (const uint32_t *)(a & ~(uintptr_t)3);
      const unsigned sh = (unsigned)(a & 3) * 8;
      const int rsw = rs >> 2;
      uint32_t W[6];
#pragma unroll
      for (int m = 0; m < 6; m++) W[m] = __funnelshift_r(TB_LDG(wq + m * rsw), TB_LDG(wq + m * rsw + 1), sh);
      int v[4];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const uint32_t sel = (uint32_t)k | ((uint32_t)(4 + k) << 4);
        const uint32_t t01 = __byte_perm(W[0], W[1], sel), t23 = __byte_perm(W[2], W[3], sel), t45 = __byte_perm(W[4], W[5], sel);
        v[k] = dp4a_us(__byte_perm(t01, t23, 0x5410), tlo, dp4a_us(t45, thi, 32)) >> 6;  // thi has zero taps on the two upper bytes
      }
      const uint32_t pk = pack_sat_u8x4(v[0], v[1], v[2], v[3]);
      if (r < h) aV0 += __vsadu4(TB_LDG((const uint32_t *)(ob + r * os + 4 * st)), pk);
      if (r > 0) aV1 += __vsadu4(TB_LDG((const uint32_t *)(ob + (r - 1) * os + 4 * st)), pk);
    }
  }
  // ---- C pass: plane rows r = 0 .. h, plane columns 4 s .. 4 s + 4
  {
    const uint32_t a_lo = 0x01010000u, b_lo = 0x02020100u, b_hi = 0x00000001u;
    for (int u = lane; u < (h + 1) * ns; u += 32) {
      const int r = u >> lns, st = u & (ns - 1);
      const uint8_t *p = rb + r * rs + 4 * st - 2;
      int acc[5] = {8, 8, 8, 8, 8};
      uint32_t b0, b1, b2;
      row12_u8(p - rs, b0, b1, b2);
#pragma unroll
      for (int k = 0; k < 5; k++) acc[k] = dp4a_us(k < 4 ? __funnelshift_r(b0, b1, 8 * k) : b1, a_lo, acc[k]);
      row12_u8(p + 2 * rs, b0, b1, b2);
#pragma unroll
      for (int k = 0; k < 5; k++) acc[k] = dp4a_us(k < 4 ? __funnelshift_r(b0, b1, 8 * k) : b1, a_lo, acc[k]);
#pragma unroll
      for (int rr = 0; rr < 2; rr++) {
        row12_u8(p + rr * rs, b0, b1, b2);
#pragma unroll
        for (int k = 0; k < 5; k++)
          acc[k] = dp4a_us(k < 4 ? __funnelshift_r(b0, b1, 8 * k) : b1, b_lo, dp4a_us(k < 4 ? __funnelshift_r(b1, b2, 8 * k) : b2, b_hi, acc[k]));
      }
      // (s + 8) >> 4 <= 255: plain byte packing
      const uint32_t q0 = (uint32_t)(acc[0] >> 4), q1 = (uint32_t)(acc[1] >> 4), q2 = (uint32_t)(acc[2] >> 4), q3 = (uint32_t)(acc[3] >> 4), q4 = (uint32_t)(acc[4] >> 4);
      const uint32_t pk0 = q0 | (q1 << 8) | (q2 << 16) | (q3 << 24), pk1 = q1 | (q2 << 8) | (q3 << 16) | (q4 << 24);
      if (r < h) {
        const uint32_t ow = TB_LDG((const uint32_t *)(ob + r * os + 4 * st));
        aC00 += __vsadu4(ow, pk0);
        aC01 += __vsadu4(ow, pk1);
      }
      if (r > 0) {
        const uint32_t ow = TB_LDG((const uint32_t *)(ob + (r - 1) * os + 4 * st));
        aC10 += __vsadu4(ow, pk0);
        aC11 += __vsadu4(ow, pk1);
      }
    }
  }
  aH0 = __reduce_add_sync(FULL, aH0); aH1 = __reduce_add_sync(FULL, aH1); aV0 = __reduce_add_sync(FULL, aV0); aV1 = __reduce_add_sync(FULL, aV1);
  aC00 = __reduce_add_sync(FULL, aC00); aC01 = __reduce_add_sync(FULL, aC01); aC10 = __reduce_add_sync(FULL, aC10); aC11 = __reduce_add_sync(FULL, aC11);
  if (cls == 0) return ho ? aH1 : aH0;
  if (cls == 1) return vo ? aV1 : aV0;
  return vo ? (ho ? aC11 : aC10) : (ho ? aC01 : aC00);
}

// ---------------------------------------------------------------------------------------------------------------
// a4: bilinear sub-pel SAD approximations.  enc/encode_block.c:174-283 and :286-414.
// up = (a+b+1)>>1, dn = (a+b)>>1.  Results: acc[0..7] in the reference's comparison order.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int up2(int a, int b) { return (a + b + 1) >> 1; }
__device__ __forceinline__ int dn2(int a, int b) { return (a + b) >> 1; }

// order: top, down, right, left, tl, tr, br, bl
template <class S>
__device__ __noinline__ uint32_t warp_sad_fasthalf(const S *a, int as, const S *b, int bs, int w, int h, int &bx, int &by) {
  uint32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const int lw = ilog2(w);
  for (int p = lane_id(); p < (h << lw); p += 32) {
    int row = p >> lw, col = p & (w - 1);
    const S *r = b + row * bs + col;
    int o = a[row * as + col];
#define PX(dy, dx) ((int)r[(dy) * bs + (dx)])
    int hL = up2(PX(0, -1), PX(0, 0)), hR = up2(PX(0, 0), PX(0, 1));
    int hLu = up2(PX(-1, -1), PX(-1, 0)), hRu = up2(PX(-1, 0), PX(-1, 1));
    int hLd = up2(PX(1, -1), PX(1, 0)), hRd = up2(PX(1, 0), PX(1, 1));
    int vUm = up2(PX(-2, -1), PX(1, -1)), vU0 = up2(PX(-2, 0), PX(1, 0)), vUp = up2(PX(-2, 1), PX(1, 1));
    int vDm = up2(PX(-1, -1), PX(2, -1)), vD0 = up2(PX(-1, 0), PX(2, 0)), vDp = up2(PX(-1, 1), PX(2, 1));
    int wLu = up2(PX(-1, -2), PX(-1, 1)), wL0 = up2(PX(0, -2), PX(0, 1)), wLd = up2(PX(1, -2), PX(1, 1));
    int wRu = up2(PX(-1, -1), PX(-1, 2)), wR0 = up2(PX(0, -1), PX(0, 2)), wRd = up2(PX(1, -1), PX(1, 2));
    int ptl = dn2(dn2(dn2(vUm, vU0), dn2(wLu, wL0)), dn2(hLu, hL));
    int ptr = dn2(dn2(dn2(vU0, vUp), dn2(wR0, wRu)), dn2(hRu, hR));
    int pbl = dn2(dn2(dn2(vD0, vDm), dn2(wL0, wLd)), dn2(hLd, hL));
    int pbr = dn2(dn2(dn2(vD0, vDp), dn2(wR0, wRd)), dn2(hR, hRd));
    acc[0] += iabs(o - up2(PX(0, 0), PX(-1, 0)));
    acc[1] += iabs(o - up2(PX(0, 0), PX(1, 0)));
    acc[2] += iabs(o - hR);
    acc[3] += iabs(o - hL);
    acc[4] += iabs(o - ptl);
    acc[5] += iabs(o - ptr);
    acc[6] += iabs(o - pbr);
    acc[7] += iabs(o - pbl);
#undef PX
  }
  const int8_t xs[8] = {0, 0, 2, -2, -2, 2, 2, -2}, ys[8] = {-2, 2, 0, 0, -2, -2, 2, 2};
  uint32_t best = 0;
  int bi = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint32_t s = warp_sum(acc[k]);
    if (k == 0 || s < best) { best = s; bi = k; }
  }
  bx = xs[bi];
  by = ys[bi];
  return best;
}

// order: top, tl, tr, left, right, bl, down, br.  fx, fy: half-pel offset found so far (selects the formula set)
template <class S>
__device__ __noinline__ uint32_t warp_sad_fastquarter(const S *o, int os, const S *r, int rs, int w, int h, int fx, int fy, int &bx, int &by) {
  uint32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const int lw = ilog2(w);
  for (int p = lane_id(); p < (h << lw); p += 32) {
    int row = p >> lw, col = p & (w - 1);
    const S *q = r + row * rs + col;
    int org = o[row * os + col];
    int a = q[0], d = q[1], f = q[rs], e = q[rs + 1];
    int vtop, vtl, vtr, vleft, vright, vbl, vdown, vbr;
    if (fx & fy) {
      int ad = up2(a, d), de = up2(d, e), af = up2(a, f), fe = up2(f, e);
      vtl = dn2(ad, af); vtop = dn2(de, a); vtr = dn2(ad, de); vleft = dn2(ad, f);
      vright = dn2(ad, e); vbl = dn2(af, fe); vdown = dn2(de, f); vbr = dn2(de, fe);
    } else if (fx) {
      int b = q[-rs], c = q[-rs + 1];
      int ad = up2(a, d), de = up2(d, e), dc = up2(d, c), af = up2(a, f), ab = up2(a, b);
      vtl = dn2(ad, ab); vtop = dn2(dc, a); vtr = dn2(ad, dc); vleft = dn2(ad, a);
      vright = dn2(ad, d); vbl = dn2(ad, af); vdown = dn2(af, d); vbr = dn2(ad, de);
    } else if (fy) {
      int g = q[rs - 1], hh = q[-1];
      int ad = up2(a, d), af = up2(a, f), fe = up2(f, e), ah = up2(a, hh), gf = up2(g, f);
      vtl = dn2(ah, af); vtop = dn2(af, a); vtr = dn2(ad, af); vleft = dn2(gf, a);
      vright = dn2(ad, f); vbl = dn2(af, gf); vdown = dn2(af, f); vbr = dn2(af, fe);
    } else {
      int b = q[-rs], hh = q[-1];
      int ad = up2(a, d), af = up2(a, f), ah = up2(a, hh), ab = up2(a, b);
      vtl = dn2(ah, ab); vtop = dn2(ab, a); vtr = dn2(ad, ab); vleft = dn2(ah, a);
      vright = dn2(ad, a); vbl = dn2(ah, af); vdown = dn2(af, a); vbr = dn2(af, ad);
    }
    acc[0] += iabs(org - vtop);   acc[1] += iabs(org - vtl);
    acc[2] += iabs(org - vtr);    acc[3] += iabs(org - vleft);
    acc[4] += iabs(org - vright); acc[5] += iabs(org - vbl);
    acc[6] += iabs(org - vdown);  acc[7] += iabs(org - vbr);
  }
  const int8_t xs[8] = {0, -1, 1, -1, 1, -1, 0, 1}, ys[8] = {-1, -1, -1, 0, 0, 1, 1, 1};
  uint32_t best = 0;
  int bi = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    uint32_t s = warp_sum(acc[k]);
    if (k == 0 || s < best) { best = s; bi = k; }
  }
  bx = xs[bi];
  by = ys[bi];
  return best;
}

// ---------------------------------------------------------------------------------------------------------------
// a5: motion_estimate.  enc/encode_block.c:517-711.  One warp runs one search; every stage evaluates its probes
// in parallel across lanes and picks the winner with the reference's sequential tie rule (first strict minimum).
// ---------------------------------------------------------------------------------------------------------------
// sub-pel probe offsets in visiting order (enc/encode_block.c:627-628, 648-649)
__constant__ int8_t c_hm[9] = {0, 0, -2, 2, 0, -2, -2, 2, 2}, c_hn[9] = {0, -2, 0, 0, 2, -2, 2, -2, 2};
__constant__ int8_t c_qm[9] = {0, 0, -1, 1, 0, -1, -1, 1, 1}, c_qn[9] = {0, -1, 0, 0, 1, -1, 1, -1, 1};
struct MeCtx {
  int size, width, height, sign, s, xpos, ypos, fw, fh, bitdepth, speed, bip;
  int mvpx, mvpy;
  double lambda;
  // work counters for the roofline (not part of the result): integer-position block SADs and sub-pel probes
  unsigned n_int, n_sub;
#if TB_ME_STAGE_PROF
  long long cyc[5];   // cycles in telescope / candidates / hexagon / half-pel / quarter-pel (diagnostics of the RD loop)
#endif
};
#if TB_ME_STAGE_PROF
#define ME_STAGE_T0() long long me_t__ = clock64()
#define ME_STAGE(k) do { const long long n__ = clock64(); c.cyc[k] += n__ - me_t__; me_t__ = n__; } while (0)
#else
#define ME_STAGE_T0() do {} while (0)
#define ME_STAGE(k) do {} while (0)
#endif

// first-minimum over lanes < n of key (cost); returns winning lane (or -1 if n == 0) and its cost
__device__ __forceinline__ int warp_first_min(uint32_t cost, int n, uint32_t &best) {
  uint32_t c = lane_id() < n ? cost : 0xffffffffu;
  uint32_t m = __reduce_min_sync(FULL, c);
  unsigned who = __ballot_sync(FULL, c == m && lane_id() < n);
  best = m;
  return who ? __ffs(who) - 1 : -1;
}

// A team of TW warps (TW == 1, or the whole CTA) runs one search: every warp executes the same control flow on the same
// totals and evaluates the SADs of its own band of h / TW rows; MeTeam::sum adds the per-lane partial SADs of the bands through
// shared memory (two alternating buffers, one __syncthreads per exchange).
template <int TW> struct MeTeam {
  uint32_t *xch;  // [2][TW][32]
  int warp, phase;
  __device__ __forceinline__ uint32_t sum(uint32_t v) {
    if (TW == 1) return v;
    uint32_t *b = xch + (phase & 1) * TW * 32;
    phase++;
    b[warp * 32 + lane_id()] = v;
    __syncthreads();
    uint32_t t = 0;
#pragma unroll
    for (int k = 0; k < TW; k++) t += b[k * 32 + lane_id()];
    return t;
  }
};

template <class S, int TW>
__device__ void warp_motion_estimate(const S *orig_full, int os, const S *ref_full, int rs, MeCtx &c, int mvcx, int mvcy, const int16_t *cand,
                                     int ncand, int &out_mvx, int &out_mvy, uint32_t &out_cost, MeTeam<TW> &tm) {
  const int lane = lane_id();
  const int band_h = c.height / TW, row0 = tm.warp * band_h;  // this warp's rows
  const S *orig = orig_full + row0 * os, *ref = ref_full + row0 * rs;
  const int s = c.s, shift = c.bitdepth - 8;
  uint32_t min_sad = 1u << 31;  // MAX_UINT32, common/global.h:63
  int optx = 0, opty = 0;
  int refx = ((mvcx + 2) >> 2) << 2, refy = ((mvcy + 2) >> 2) << 2;
  refx = (int)(int16_t)refx;
  refy = (int)(int16_t)refy;

  ME_STAGE_T0();
  // ---- telescope search: 5x5 grids at steps 32,16,8,4 quarter-pels (:531-561)
  if ((c.size == 16 && c.bip) || c.speed == 0) {
    for (int step = 32; step >= 4; step >>= 1) {
      // sequential visiting order: k (y) outer, l (x) inner; the centre is skipped for step < 32
      int idx = lane;
      if (step < 32 && idx >= 12) idx++;  // 24 probes, hole at grid index 12
      int n = step < 32 ? 24 : 25;
      int k = (idx / 5 - 2) * step, l = (idx % 5 - 2) * step;
      int cx = (int)(int16_t)(refx + l), cy = (int)(int16_t)(refy + k);
      clip_mv(cx, cy, c.ypos, c.xpos, c.fw, c.fh, c.size, c.size, c.sign);
      uint32_t sad;
      if (step == 32 && c.size == 16 && c.speed == 1) {
        // widesad at every grid point: best of x offsets -3,-1,0,1,3 (first minimum), enc/encode_block.c:430-453
        const int offs[5] = {-3, -1, 0, 1, 3};
        uint32_t b = 0xffffffffu;
        int bxo = 0;
        int base = s * (cx >> 2) + s * (cy >> 2) * rs;
#pragma unroll
        for (int t = 0; t < 5; t++) {
          uint32_t v = tm.sum(multi_sad<S, TW>(orig, os, ref, rs, c.width, band_h, base + offs[t], n));
          if (v < b) { b = v; bxo = offs[t]; }
        }
        sad = b;
        cx = (int)(int16_t)(cx + (s * bxo << 2));
        c.n_int += 5 * n;
      } else {
        sad = tm.sum(multi_sad<S, TW>(orig, os, ref, rs, c.width, band_h, s * (cx >> 2) + s * (cy >> 2) * rs, n));
        c.n_int += n;
      }
      uint32_t cost = (sad >> shift) + mv_cost(c.lambda, quote_mv_bits(cy - c.mvpy, cx - c.mvpx));
      uint32_t best;
      int w = warp_first_min(cost, n, best);
      if (best < min_sad) {
        min_sad = best;
        optx = __shfl_sync(FULL, cx, w);
        opty = __shfl_sync(FULL, cy, w);
      }
      refx = optx;
      refy = opty;
    }
  }

  ME_STAGE(0);
  // ---- candidate search (:564-581); 16x16 blocks use the five-position wide SAD
  for (int base = 0; base < ncand; base += 32) {
    int n = min(32, ncand - base);
    int cx = 0, cy = 0;
    if (lane < n) {
      cx = (int)(int16_t)(cand[2 * (base + lane)] << 2);
      cy = (int)(int16_t)(cand[2 * (base + lane) + 1] << 2);
    }
    clip_mv(cx, cy, c.ypos, c.xpos, c.fw, c.fh, c.size, c.size, c.sign);
    uint32_t sad;
    int pos = s * (cx >> 2) + s * (cy >> 2) * rs;
    if (c.size == 16) {
      const int offs[5] = {-3, -1, 0, 1, 3};
      uint32_t b = 0xffffffffu;
      int bxo = 0;
#pragma unroll
      for (int t = 0; t < 5; t++) {
        uint32_t v = tm.sum(multi_sad<S, TW>(orig, os, ref, rs, c.width, band_h, pos + offs[t], n));
        if (v < b) { b = v; bxo = offs[t]; }
      }
      sad = b;
      cx = (int)(int16_t)(cx + (s * bxo << 2));
      c.n_int += 5 * n;
    } else {
      sad = tm.sum(multi_sad<S, TW>(orig, os, ref, rs, c.width, band_h, pos, n));
      c.n_int += n;
    }
    uint32_t cost = (sad >> shift) + mv_cost(c.lambda, quote_mv_bits(cy - c.mvpy, cx - c.mvpx));
    uint32_t best;
    int w = warp_first_min(cost, n, best);
    if (w >= 0 && best < min_sad) {
      min_sad = best;
      optx = __shfl_sync(FULL, cx, w);
      opty = __shfl_sync(FULL, cy, w);
    }
  }
  refx = optx;
  refy = opty;

  ME_STAGE(1);
  // ---- hexagon refinement (:583-616): visit dir = start..end cyclically; first strict minimum wins
  {
    const int maxsteps = (c.size <= 16 || c.speed == 0) ? 6 : 0;
    int start = 0, end = 5;
    for (int step = 1; step < maxsteps; step++) {
      const int diy[6] = {1, 2, 1, -1, -2, -1}, dix[6] = {-1, 0, 1, 1, 0, -1};
      int n = ((end - start + 6) % 6) + 1;  // number of directions visited
      int dir = (start + lane) % 6;
      int cx = (int)(int16_t)(refx + diy[dir] * 4), cy = (int)(int16_t)(refy + dix[dir] * 4);
      clip_mv(cx, cy, c.ypos, c.xpos, c.fw, c.fh, c.size, c.size, c.sign);
      uint32_t sad = tm.sum(multi_sad<S, TW>(orig, os, ref, rs, c.width, band_h, s * (cx >> 2) + s * (cy >> 2) * rs, n));
      c.n_int += n;
      uint32_t cost = (sad >> shift) + mv_cost(c.lambda, quote_mv_bits(cy - c.mvpy, cx - c.mvpx));
      uint32_t best;
      int w = warp_first_min(cost, n, best);
      int best_dir = -1;
      if (best < min_sad) {
        min_sad = best;
        optx = __shfl_sync(FULL, cx, w);
        opty = __shfl_sync(FULL, cy, w);
        best_dir = (start + w) % 6;
      }
      refx = optx;
      refy = opty;
      start = best_dir ? best_dir - 1 : 5;
      end = start + 2;
      end -= (end >= 6) * 6;
      if (best_dir < 0) break;
    }
  }

  ME_STAGE(2);
  int ydh = 0, xdh = 0, ydq = 0, xdq = 0;
  uint32_t cmin = min_sad;
  c.n_sub += c.speed == 0 ? 16 : 2;
  if (c.speed == 0) {
    // ---- true half-pel then quarter-pel probes (:625-663)
    const int8_t *hm = c_hm, *hn = c_hn, *qm = c_qm, *qn = c_qn;
    // each stage: the eight probes are evaluated together; the winner is then chosen in the reference's sequential order
    // (strict '<', i = 1..8).  The cost of probe i is left on lane i - 1.
    for (int stage = 0; stage < 2; stage++) {
      const int8_t *dm = stage ? qm : hm, *dn = stage ? qn : hn;
      const int bx = optx, by = opty;
      uint32_t sad = 0xffffffffu;
      if (sizeof(S) == 1 && stage == 0 && !((bx | by) & 3))
        sad = halfpel_stage_sads_u8((const uint8_t *)orig_full, os, (const uint8_t *)ref_full, rs, c.width, c.height, bx, by, dn, dm, c.sign, c.bip, c.fw, c.fh, c.xpos, c.ypos,
                                    row0, band_h);
      const int i1 = (lane & 7) + 1;
      const int cy = (int)(int16_t)(by + dm[i1]), cx = (int)(int16_t)(bx + dn[i1]);
      if (sad == 0xffffffffu) {  // 16-bit samples, the quarter-pel stage, or a geometry halfpel_stage_sads_u8 does not take: one probe per 4-lane group
        const int tq = (lane >> 2) + 1;
        const int qy = (int)(int16_t)(by + dm[tq]), qx = (int)(int16_t)(bx + dn[tq]);
        sad = subpel_stage_sads<S>(orig_full, os, ref_full, rs, c.width, c.height, qx, qy, c.sign, c.bip, c.fw, c.fh, c.xpos, c.ypos, c.bitdepth, row0, band_h);
        sad = __shfl_sync(FULL, sad, (lane & 7) * 4);
      }
      sad = tm.sum(sad);
      const uint32_t cost = (sad >> shift) + mv_cost(c.lambda, quote_mv_bits(cy - c.mvpy, cx - c.mvpx));
      int yd = 0, xd = 0;
      for (int i = 1; i <= 8; i++) {
        uint32_t ci = __shfl_sync(FULL, cost, i - 1);
        if (ci < cmin) { cmin = ci; yd = dm[i]; xd = dn[i]; }
      }
      if (stage == 0) {
        ydh = yd; xdh = xd;
        optx = (int)(int16_t)(optx + xdh);
        opty = (int)(int16_t)(opty + ydh);
      } else {
        ydq = yd; xdq = xd;
      }
      ME_STAGE(3 + stage);
    }
  } else {
    // ---- bilinear approximations (:664-703)
    int rx = (int)(int16_t)(refx * s), ry = (int)(int16_t)(refy * s);
    int spx, spy;
    uint32_t sad = warp_sad_fasthalf<S>(orig_full, os, ref_full + (rx >> 2) + (ry >> 2) * rs, rs, c.width, c.height, spx, spy);
    uint32_t cost = (sad >> shift) + mv_cost(c.lambda, quote_mv_bits(ry + s * spy - c.mvpy, rx + s * spx - c.mvpx));
    if (cost < cmin) { cmin = cost; xdh = s * spx; ydh = s * spy; }
    spx = xdh;
    spy = ydh;
    rx = (int)(int16_t)(optx + s * spx);
    ry = (int)(int16_t)(opty + s * spy);
    optx = (int)(int16_t)(optx + xdh);
    opty = (int)(int16_t)(opty + ydh);
    int qx, qy;
    sad = warp_sad_fastquarter<S>(orig_full, os, ref_full + s * (rx >> 2) + s * (ry >> 2) * rs, rs, c.width, c.height, spx, spy, qx, qy);
    cost = (sad >> shift) + mv_cost(c.lambda, quote_mv_bits(ry + s * qy - c.mvpy, rx + s * qx - c.mvpx));
    if (cost < cmin) { cmin = cost; xdq = s * qx; ydq = s * qy; }
  }
  out_mvx = (int)(int16_t)(optx + xdq);
  out_mvy = (int)(int16_t)(opty + ydq);
  out_cost = cmin < min_sad ? cmin : min_sad;
}

// ---------------------------------------------------------------------------------------------------------------
// a5 for small blocks: FOUR searches per warp, eight lanes each.  A search over a block of <= 64 samples spends most of its
// instructions in stages that can use only 3-8 lanes (candidate list, hexagon rounds, the eight sub-pel probes) and in per-stage
// scalar work (clipping, pricing, winner selection); sharing the warp between four searches issues that work once for four
// (profiles/r1_ncu_summary.md section E: 4.2 k warp instructions per search, a third of the stalls are instruction fetches).
// Every lane of a group carries its search's state; all collectives use the group's 8-lane mask, so groups diverge freely.
// Same stages, visiting order and tie rules as warp_motion_estimate (8-bit samples, speed 0).
// ---------------------------------------------------------------------------------------------------------------
struct QuadItem {
  const uint8_t *orig, *ref;
  const int16_t *cand;
  double lambda;
  int os, rs, size, w, h, sign, xpos, ypos, mvpx, mvpy, mvcx, mvcy, ncand;
};
__device__ __forceinline__ int group_first_min(unsigned gm, uint32_t cost, bool valid, uint32_t &best) {  // lowest lane among the minima; -1 if none valid
  const uint32_t c = valid ? cost : 0xffffffffu;
  best = __reduce_min_sync(gm, c);
  const unsigned who = __ballot_sync(gm, valid && c == best);
  return who ? __ffs(who) - 1 : -1;
}
__device__ __noinline__ void quad_motion_estimate(const QuadItem &q, int fw, int fh, int bip, int &out_mvx, int &out_mvy, uint32_t &out_cost, unsigned &n_int) {
  const int lane = lane_id(), gl = lane & 7, g0 = lane & 24;
  const unsigned gm = 0xffu << g0;
  const int s = q.sign ? -1 : 1;
  uint32_t min_sad = 1u << 31;
  int optx = 0, opty = 0;
  int refx = (int)(int16_t)(((q.mvcx + 2) >> 2) << 2), refy = (int)(int16_t)(((q.mvcy + 2) >> 2) << 2);
  n_int = 0;
  // SAD + rate of one integer position (this lane's probe)
  auto int_cost = [&](int cx, int cy, uint32_t &sad_out) {
    const uint8_t *r = q.ref + s * (cx >> 2) + s * (cy >> 2) * q.rs;
    sad_out = sad_partial<uint8_t>(q.orig, q.os, r, q.rs, q.w, q.h, 0, 1);
  };
  // ---- telescope (:531-561): 25 / 24 grid points per step, eight per pass; a lane keeps its earliest minimum, the group then takes the
  // smallest cost and, among equal costs, the earliest visiting index
  for (int step = 32; step >= 4; step >>= 1) {
    const int n = step < 32 ? 24 : 25;
    uint32_t bc = 0xffffffffu;
    int bidx = 64, bx = 0, by = 0;
    for (int pass = 0; pass < 4; pass++) {
      const int vi = pass * 8 + gl;
      if (vi < n) {
        int idx = vi;
        if (step < 32 && idx >= 12) idx++;
        int cx = (int)(int16_t)(refx + (idx % 5 - 2) * step), cy = (int)(int16_t)(refy + (idx / 5 - 2) * step);
        clip_mv(cx, cy, q.ypos, q.xpos, fw, fh, q.size, q.size, q.sign);
        uint32_t sad;
        int_cost(cx, cy, sad);
        const uint32_t c = sad + mv_cost(q.lambda, quote_mv_bits(cy - q.mvpy, cx - q.mvpx));
        if (c < bc) { bc = c; bidx = vi; bx = cx; by = cy; }
      }
    }
    n_int += n;
    const uint32_t m = __reduce_min_sync(gm, bc);
    const unsigned mi = __reduce_min_sync(gm, bc == m ? (unsigned)bidx : 64u);
    const unsigned who = __ballot_sync(gm, bc == m && (unsigned)bidx == mi);
    const int wl = __ffs(who) - 1;
    const int wx = __shfl_sync(gm, bx, wl), wy = __shfl_sync(gm, by, wl);
    if (m < min_sad) { min_sad = m; optx = wx; opty = wy; }
    refx = optx;
    refy = opty;
  }
  // ---- candidates (:564-581); blocks of a 16x16 coding block use the five-position wide SAD
  for (int base = 0; base < q.ncand; base += 8) {
    const int n = min(8, q.ncand - base);
    const bool valid = gl < n;
    int cx = 0, cy = 0;
    uint32_t cost = 0;
    if (valid) {
      cx = (int)(int16_t)(q.cand[2 * (base + gl)] << 2);
      cy = (int)(int16_t)(q.cand[2 * (base + gl) + 1] << 2);
      clip_mv(cx, cy, q.ypos, q.xpos, fw, fh, q.size, q.size, q.sign);
      uint32_t sad;
      if (q.size == 16) {
        const int offs[5] = {-3, -1, 0, 1, 3};
        const uint8_t *r = q.ref + s * (cx >> 2) + s * (cy >> 2) * q.rs;
        uint32_t b = 0xffffffffu;
        int bxo = 0;
#pragma unroll
        for (int t = 0; t < 5; t++) {
          const uint32_t v = sad_partial<uint8_t>(q.orig, q.os, r + offs[t], q.rs, q.w, q.h, 0, 1);
          if (v < b) { b = v; bxo = offs[t]; }
        }
        sad = b;
        cx = (int)(int16_t)(cx + (s * bxo << 2));
      } else
        int_cost(cx, cy, sad);
      cost = sad + mv_cost(q.lambda, quote_mv_bits(cy - q.mvpy, cx - q.mvpx));
    }
    n_int += (q.size == 16 ? 5 : 1) * n;
    uint32_t best;
    const int wl = group_first_min(gm, cost, valid, best);
    const int wx = __shfl_sync(gm, cx, wl < 0 ? g0 : wl), wy = __shfl_sync(gm, cy, wl < 0 ? g0 : wl);
    if (wl >= 0 && best < min_sad) { min_sad = best; optx = wx; opty = wy; }
  }
  refx = optx;
  refy = opty;
  // ---- hexagon refinement (:583-616)
  {
    int start = 0, end = 5;
    for (int step = 1; step < 6; step++) {
      const int diy[6] = {1, 2, 1, -1, -2, -1}, dix[6] = {-1, 0, 1, 1, 0, -1};
      const int n = ((end - start + 6) % 6) + 1;
      const bool valid = gl < n;
      const int dir = (start + gl) % 6;
      int cx = (int)(int16_t)(refx + diy[dir] * 4), cy = (int)(int16_t)(refy + dix[dir] * 4);
      uint32_t cost = 0;
      if (valid) {
        clip_mv(cx, cy, q.ypos, q.xpos, fw, fh, q.size, q.size, q.sign);
        uint32_t sad;
        int_cost(cx, cy, sad);
        cost = sad + mv_cost(q.lambda, quote_mv_bits(cy - q.mvpy, cx - q.mvpx));
      }
      n_int += n;
      uint32_t best;
      const int wl = group_first_min(gm, cost, valid, best);
      const int wx = __shfl_sync(gm, cx, wl), wy = __shfl_sync(gm, cy, wl);
      int best_dir = -1;
      if (best < min_sad) { min_sad = best; optx = wx; opty = wy; best_dir = (start + (wl - g0)) % 6; }
      refx = optx;
      refy = opty;
      start = best_dir ? best_dir - 1 : 5;
      end = start + 2;
      end -= (end >= 6) * 6;
      if (best_dir < 0) break;
    }
  }
  // ---- half-pel, then quarter-pel probes (:625-663): probe i on lane i - 1 of the group
  int ydh = 0, xdh = 0, ydq = 0, xdq = 0;
  uint32_t cmin = min_sad;
  for (int stage = 0; stage < 2; stage++) {
    const int8_t *dm = stage ? c_qm : c_hm, *dn = stage ? c_qn : c_hn;
    const int cy = (int)(int16_t)(opty + dm[gl + 1]), cx = (int)(int16_t)(optx + dn[gl + 1]);
    int hi, vi, xf, yf;
    split_mv(cx, cy, q.sign, 2, fw, fh, q.xpos, q.ypos, q.w, q.h, hi, vi, xf, yf);
    const uint8_t *ip = q.ref + vi * q.rs + hi;
    const int RH = q.h >= 8 ? 8 : q.h, nseg = q.h / RH, units = (q.w >> 2) * nseg;
    uint32_t sad = 0;
    for (int u = 0; u < units; u++) {
      const int strip = u / nseg, seg = u - strip * nseg;
      sad += strip_sad_subpel_u8(q.orig, q.os, ip, q.rs, strip * 4, seg * RH, RH, xf, yf, bip);
    }
    const uint32_t cost = sad + mv_cost(q.lambda, quote_mv_bits(cy - q.mvpy, cx - q.mvpx));
    int yd = 0, xd = 0;
    for (int i = 1; i <= 8; i++) {
      const uint32_t ci = __shfl_sync(gm, cost, g0 + i - 1);
      if (ci < cmin) { cmin = ci; yd = dm[i]; xd = dn[i]; }
    }
    if (stage == 0) {
      ydh = yd; xdh = xd;
      optx = (int)(int16_t)(optx + xdh);
      opty = (int)(int16_t)(opty + ydh);
    } else {
      ydq = yd; xdq = xd;
    }
  }
  out_mvx = (int)(int16_t)(optx + xdq);
  out_mvy = (int)(int16_t)(opty + ydq);
  out_cost = cmin < min_sad ? cmin : min_sad;
}

// ---------------------------------------------------------------------------------------------------------------
// a5: motion_estimate_bi, simultaneous bi-directional search with mv0 = -mv1.  enc/encode_block.c:798-914.
// Each probe is SAD(orig, (P0 + P1) >> 1) with both predictions truly interpolated; up to eight probes of a step run
// concurrently on 4-lane groups, the winner is then taken in the reference's visiting order.
// ---------------------------------------------------------------------------------------------------------------
template <class S>
__device__ __noinline__ uint32_t bi_probe_sad(const S *o, int os, const S *ref0, const S *ref1, int rs, int size, int mvx0, int mvy0, int mvx1, int mvy1, int sign, int bip,
                                              int fw, int fh, int xpos, int ypos, int bitdepth) {
  int hi0, vi0, xf0, yf0, hi1, vi1, xf1, yf1;
  split_mv(mvx0, mvy0, sign, 2, fw, fh, xpos, ypos, size, size, hi0, vi0, xf0, yf0);
  split_mv(mvx1, mvy1, 1 - sign, 2, fw, fh, xpos, ypos, size, size, hi1, vi1, xf1, yf1);
  const S *ip0 = ref0 + vi0 * rs + hi0, *ip1 = ref1 + vi1 * rs + hi1;
  const int maxv = (1 << bitdepth) - 1, ls = ilog2(size), sub = lane_id() & 3;
  uint32_t acc = 0;
  for (int p = sub; p < size * size; p += 4) {
    int row = p >> ls, col = p & (size - 1);
    const S *q0 = ip0 + row * rs + col, *q1 = ip1 + row * rs + col;
    int v0 = (xf0 == 0 && yf0 == 0) ? (int)q0[0] : luma_sample<S>(q0, rs, xf0, yf0, bip, maxv);
    int v1 = (xf1 == 0 && yf1 == 0) ? (int)q1[0] : luma_sample<S>(q1, rs, xf1, yf1, bip, maxv);
    acc += (uint32_t)iabs((int)o[row * os + col] - ((v0 + v1) >> 1));
  }
  return group_sum(acc, 4);
}

// The same with the whole warp on ONE probe (blocks >= 16x16 inside the device RD loop): integer positions are averaged and compared as 32-bit words
// straight from the reference frames (lanes along the row); any other position is interpolated once per reference by the prediction routine
// (warp_interp: DP4A strips) into the caller's two scratch blocks (pitch = size) and compared as words from there.
template <class S>
__device__ __noinline__ uint32_t bi_probe_sad_warp(const S *o, int os, const S *ref0, const S *ref1, int rs, int size, int mvx0, int mvy0, int mvx1, int mvy1, int sign, int bip,
                                                   int fw, int fh, int xpos, int ypos, int bitdepth, S *s0, S *s1) {
  constexpr int PW = Word<S>::PW;
  int hi0, vi0, xf0, yf0, hi1, vi1, xf1, yf1;
  split_mv(mvx0, mvy0, sign, 2, fw, fh, xpos, ypos, size, size, hi0, vi0, xf0, yf0);
  split_mv(mvx1, mvy1, 1 - sign, 2, fw, fh, xpos, ypos, size, size, hi1, vi1, xf1, yf1);
  const S *p0 = ref0 + vi0 * rs + hi0, *p1 = ref1 + vi1 * rs + hi1;
  int st0 = rs, st1 = rs;
  if (xf0 | yf0) { __syncwarp(); warp_interp<S>(s0, size, ref0, rs, size, size, mvx0, mvy0, sign, 0, bip, fw, fh, xpos, ypos, bitdepth); p0 = s0; st0 = size; }
  if (xf1 | yf1) { __syncwarp(); warp_interp<S>(s1, size, ref1, rs, size, size, mvx1, mvy1, 1 - sign, 0, bip, fw, fh, xpos, ypos, bitdepth); p1 = s1; st1 = size; }
  __syncwarp();
  const int lane = lane_id(), LW = size / PW, LWe = LW < 32 ? LW : 32, RP = 32 / LWe, CI = LW / LWe;
  const int col0 = lane & (LWe - 1), rsub = lane / LWe;
  uint32_t acc = 0;
  for (int row = rsub; row < size; row += RP)
    for (int ci = 0; ci < CI; ci++) {
      const int col = (col0 + ci * 32) * PW;
      const uint32_t a = *(const uint32_t *)(o + row * os + col), r0 = ldw_any(p0 + row * st0 + col), r1 = ldw_any(p1 + row * st1 + col);
      acc += word_sad<S>(a, sizeof(S) == 1 ? __vhaddu4(r0, r1) : __vhaddu2(r0, r1));  // (v0 + v1) >> 1 per sample
    }
  __syncwarp();
  return warp_sum(acc);
}

template <class S>
__device__ void warp_motion_estimate_bi(const S *orig, int os, const S *ref0, const S *ref1, int rs, int size, int sign, int xpos, int ypos, int fw, int fh, int bitdepth, int bip,
                                        double lambda, int mvcx, int mvcy, int mvpx, int mvpy, const int16_t *cand, int ncand, int &out_mvx, int &out_mvy,
                                        uint32_t &out_cost, S *scratch0 = nullptr, S *scratch1 = nullptr) {
  const int lane = lane_id(), shift = bitdepth - 8;
  // with scratch blocks and >= 16x16: one probe at a time on the whole warp (bi_probe_sad_warp); else eight probes at a time on 4-lane groups
  const bool whole = scratch0 != nullptr && size >= 16;
  const int gl = whole ? 32 : 4, grp = lane / gl, per = 32 / gl;
  uint32_t min_sad = 1u << 31;
  int optx = 0, opty = 0;
  int refx = (int)(int16_t)(((mvcx + 2) >> 2) << 2), refy = (int)(int16_t)(((mvcy + 2) >> 2) << 2);
  // six telescope steps (3x3 grids) followed by one pass over the six candidates
  for (int stage = 0; stage < 7; stage++) {
    const int step = stage < 6 ? (32 >> stage) : 0;
    const int nslots = stage < 6 ? 9 : 6;
    for (int base = 0; base < nslots; base += per) {
      // slot handled by this lane group
      const int slot = base + grp;
      bool valid = slot < nslots;
      int cx = 0, cy = 0;
      if (valid) {
        if (stage < 6) {
          int k = (slot / 3 - 1) * step, l = (slot % 3 - 1) * step;
          if (step < 32 && k == 0 && l == 0) valid = false;
          if (step == 1) {
            int vf = refy & 3, hf = refx & 3;
            bool ex = (vf == 0 && hf == 0) ? (iabs(k) != iabs(l)) : ((vf == 2 && hf == 2) ? true : (iabs(k) == iabs(l)));
            if (ex) valid = false;
          }
          cy = (int)(int16_t)(refy + k);
          cx = (int)(int16_t)(refx + l);
        } else {
          if (slot < 4) { if (slot < ncand) { cx = cand[2 * slot]; cy = cand[2 * slot + 1]; } }
          else if (slot == 4) { cx = mvpx; cy = mvpy; }
        }
      }
      int c0x = cx, c0y = cy;
      clip_mv(c0x, c0y, ypos, xpos, fw, fh, size, size, sign);
      int c1x = c0x, c1y = c0y;  // the second clip runs on the already clipped vector; its result is the one kept
      clip_mv(c1x, c1y, ypos, xpos, fw, fh, size, size, 1 - sign);
      uint32_t sad = 0;
      if (!whole) sad = bi_probe_sad<S>(orig, os, ref0, ref1, rs, size, c0x, c0y, c1x, c1y, sign, bip, fw, fh, xpos, ypos, bitdepth);
      else if (valid) sad = bi_probe_sad_warp<S>(orig, os, ref0, ref1, rs, size, c0x, c0y, c1x, c1y, sign, bip, fw, fh, xpos, ypos, bitdepth, scratch0, scratch1);  // warp-uniform
      uint32_t cost = (sad >> shift) + mv_cost(lambda, quote_mv_bits((int)(int16_t)(c1y - mvpy), (int)(int16_t)(c1x - mvpx)));
      for (int t = 0; t < per; t++) {
        bool v = __shfl_sync(FULL, (int)valid, t * gl) != 0;
        uint32_t ct = __shfl_sync(FULL, cost, t * gl);
        int tx = __shfl_sync(FULL, c1x, t * gl), ty = __shfl_sync(FULL, c1y, t * gl);
        if (v && ct < min_sad) { min_sad = ct; optx = tx; opty = ty; }
      }
    }
    if (stage < 6) { refx = optx; refy = opty; }
  }
  out_mvx = optx;
  out_mvy = opty;
  out_cost = min_sad;
}

// ---------------------------------------------------------------------------------------------------------------
// a10/a11: integer DCT.  common/transform.c:245-308 (forward), :411-494 (inverse).
// Matrix M_N[i][j] = +-T[fold((2j+1)*i*32/N mod 128)] (HEVC core transform); kept in constant memory because every
// lane of a warp reads the same coefficient in the inner loops (broadcast).
// ---------------------------------------------------------------------------------------------------------------
__constant__ int8_t c_T[33] = {64, 90, 90, 90, 89, 88, 87, 85, 83, 82, 80, 78, 75, 73, 70, 67, 64,
                               61, 57, 54, 50, 46, 43, 38, 36, 31, 25, 22, 18, 13, 9,  4,  0};
__device__ __forceinline__ int dct_coef(int lN, int i, int j) {  // N = 1 << lN
  int m = ((2 * j + 1) * i * (32 >> lN)) & 127;
  if (m > 64) m = 128 - m;
  return m > 32 ? -(int)c_T[64 - m] : (int)c_T[m];
}

// The four matrices (N = 4, 8, 16, 32) as int16 tables for shared memory: lanes of a warp read DIFFERENT coefficients
// in the transform loops, which constant memory would serialise.  Layout: N=4 @0, 8 @16, 16 @80, 32 @336 (1360 entries).
constexpr int DCT_TAB_SIZE = 1360;
__device__ __forceinline__ int dct_tab_ofs(int lN) { return lN == 2 ? 0 : (lN == 3 ? 16 : (lN == 4 ? 80 : 336)); }
// int8 tables, natural pitches: the 16/32-point rows are read with 128-bit loads that are uniform per quarter-warp (dot16_block)
constexpr int DCT_TAB8_SIZE = 16 + 64 + 16 * 16 + 32 * 32;  // 1360; every row of the 16- and 32-point tables is 16-byte aligned
__device__ __forceinline__ int dct_tab8_ofs(int lN) { return lN == 2 ? 0 : (lN == 3 ? 16 : (lN == 4 ? 80 : 336)); }
__device__ __forceinline__ int dct_tab8_pitch(int lN) { return 1 << lN; }
__device__ __forceinline__ void dct_tab_fill(int16_t *tab) {  // call with all threads of the CTA, then __syncthreads()
  for (int t = threadIdx.x; t < DCT_TAB_SIZE; t += blockDim.x) {
    int lN = t < 16 ? 2 : (t < 80 ? 3 : (t < 336 ? 4 : 5));
    int e = t - dct_tab_ofs(lN);
    tab[t] = (int16_t)dct_coef(lN, e >> lN, e & ((1 << lN) - 1));
  }
}

// int8 forms (all coefficients are within +-90) for the DP2A inner loops: tab8[ofs + i*N + k] = M[i][k] and
// tab8t[ofs + j*N + k] = M[k][j]; every row starts 4-byte aligned.
__device__ __forceinline__ void dct_tab8_fill(int8_t *tab8, int8_t *tab8t) {
  for (int t = threadIdx.x; t < DCT_TAB_SIZE; t += blockDim.x) {
    int lN = t < 16 ? 2 : (t < 80 ? 3 : (t < 336 ? 4 : 5));
    int e = t - dct_tab_ofs(lN), i = e >> lN, k = e & ((1 << lN) - 1);
    int d = dct_tab8_ofs(lN) + i * dct_tab8_pitch(lN) + k;
    tab8[d] = (int8_t)dct_coef(lN, i, k);
    tab8t[d] = (int8_t)dct_coef(lN, k, i);
  }
}
// sum += m[0..n) . v[0..n)  (m: int8 row, v: int16 row, both 4-byte aligned, n a multiple of 4): two DP2A per four terms
__device__ __forceinline__ int dot_s8_s16(const int8_t *m, const int16_t *v, int n) {
  int sum = 0;
  const uint32_t *mw = (const uint32_t *)m, *vw = (const uint32_t *)v;
  for (int k = 0; k < (n >> 2); k++) {
    uint32_t mm = mw[k];
    sum = __dp2a_lo((int)vw[2 * k], (int)mm, sum);
    sum = __dp2a_hi((int)vw[2 * k + 1], (int)mm, sum);
  }
  return sum;
}

// acc[r][c] += A_r[0..16) . B_c[0..16): RA rows of an int8 matrix (stride sa bytes) against RB int16 vectors (stride sb elements),
// 16 terms each.  Every operand row is fetched once with 128-bit shared loads (rows 16-byte aligned) and used RA (RB) times:
// (RA + 2 RB) loads for 8 RA RB DP2A instead of 12 loads per 8 DP2A in the one-output-at-a-time form.
template <int RA, int RB>
__device__ __forceinline__ void dot16_block(const int8_t *A, int sa, const int16_t *B, int sb, int (&acc)[RA][RB]) {
  uint4 a[RA];
#pragma unroll
  for (int r = 0; r < RA; r++) a[r] = *(const uint4 *)(A + r * sa);
#pragma unroll
  for (int c = 0; c < RB; c++) {
    const uint4 b0 = *(const uint4 *)(B + c * sb), b1 = *(const uint4 *)(B + c * sb + 8);
#pragma unroll
    for (int r = 0; r < RA; r++) {
      int t = acc[r][c];
      t = __dp2a_lo((int)b0.x, (int)a[r].x, t); t = __dp2a_hi((int)b0.y, (int)a[r].x, t);
      t = __dp2a_lo((int)b0.z, (int)a[r].y, t); t = __dp2a_hi((int)b0.w, (int)a[r].y, t);
      t = __dp2a_lo((int)b1.x, (int)a[r].z, t); t = __dp2a_hi((int)b1.y, (int)a[r].z, t);
      t = __dp2a_lo((int)b1.z, (int)a[r].w, t); t = __dp2a_hi((int)b1.w, (int)a[r].w, t);
      acc[r][c] = t;
    }
  }
}

// per-warp scratch: in[32*33] + tmp[16*33] int16 (padded pitch 33 -> conflict-free column access)
struct alignas(16) TxScratch {
  alignas(16) int16_t in[48 * 40];   // forward input tile (<= 32 rows, pitch 40) / inverse: rcoeff^T (16 rows) + T^T (32 rows)
  alignas(16) int16_t tmp[16 * 40];
  int16_t cq[256];
  int16_t rc[256];
};

// Forward transform of `size` x `size` residual (row pitch = size, in global or shared memory) into sc.rc-style
// compact qsize x qsize output `coef` (pitch qsize).  Returns nothing; all lanes participate.
__device__ void warp_fwd_transform(const int16_t *block, int bpitch, int size, int fast, int bitdepth, TxScratch &sc, int16_t *coef, const int16_t *tab) {
  const int lane = lane_id();
  int size1 = size, scale = 1;
  if (size > (32 >> fast)) { size1 = 32 >> fast; scale = size / size1; }
  const int l1 = ilog2(size1), qsize = min(size, 16);
  const int16_t *M = tab + dct_tab_ofs(l1);
  // load (with box-sum down-scaling for large blocks, saturating like common/transform.c:261-278)
  for (int p = lane; p < size1 * size1; p += 32) {
    int i = p >> l1, j = p & (size1 - 1);
    int v;
    if (scale == 1) v = block[i * bpitch + j];
    else {
      int sum = 0;
      for (int m = 0; m < scale; m++)
        for (int n = 0; n < scale; n++) sum = iclip(sum + block[(i * scale + m) * bpitch + j * scale + n], -16384, 16383);
      v = sum;
    }
    sc.in[i * 33 + j] = (int16_t)v;
  }
  __syncwarp();
  const int shift1 = ilog2(size) + ilog2(scale) + bitdepth - 8, add1 = 1 << (shift1 - 1);
  const int shift2 = l1 + 5, add2 = 1 << (shift2 - 1);
  // 1st dimension: tmp[i][j] = (sum_k M[i][k] * in[j][k] + add1) >> shift1, i < qsize, j < size1
  for (int p = lane; p < qsize * size1; p += 32) {
    int i = p >> l1, j = p & (size1 - 1);
    int sum = 0;
    for (int k = 0; k < size1; k++) sum += (int)M[(i << l1) + k] * (int)sc.in[j * 33 + k];
    sc.tmp[i * 33 + j] = (int16_t)((sum + add1) >> shift1);
  }
  __syncwarp();
  // 2nd dimension: coef[i][j] = (sum_k M[i][k] * tmp[j][k] + add2) >> shift2, i, j < qsize
  const int lq = ilog2(qsize);
  for (int p = lane; p < qsize * qsize; p += 32) {
    int i = p >> lq, j = p & (qsize - 1);
    int sum = 0;
    for (int k = 0; k < size1; k++) sum += (int)M[(i << l1) + k] * (int)sc.tmp[j * 33 + k];
    coef[i * qsize + j] = (int16_t)((sum + add2) >> shift2);
  }
  __syncwarp();
}

// Inverse transform from compact qsize x qsize coefficients (pitch cpitch) to a size x size residual block
// (pitch bpitch; size <= 32 core, 64/128 by sample replication, common/transform.c:467-494).
__device__ void warp_inv_transform(const int16_t *coef, int cpitch, int size, int bitdepth, TxScratch &sc, int16_t *block, int bpitch, const int16_t *tab) {
  const int lane = lane_id();
  const int core = min(size, 32), rep = size / core, lc = ilog2(core), qsize = min(size, 16);
  const int shift2 = 20 - bitdepth, add2 = 1 << (shift2 - 1);
  const int16_t *M = tab + dct_tab_ofs(lc);
  // 1st dimension: tmp[i][j] = clip16((sum_k M[k][j] * coef[k][i] + 64) >> 7), i < qsize, j < core
  for (int p = lane; p < qsize * core; p += 32) {
    int i = p >> lc, j = p & (core - 1);
    int sum = 0;
    for (int k = 0; k < qsize; k++) sum += (int)M[(k << lc) + j] * (int)coef[k * cpitch + i];
    sc.tmp[i * 33 + j] = (int16_t)iclip((sum + 64) >> 7, -32768, 32767);
  }
  __syncwarp();
  // 2nd dimension: out[i][j] = clip16((sum_k M[k][j] * tmp[k][i] + add2) >> shift2), i, j < core
  for (int p = lane; p < core * core; p += 32) {
    int i = p >> lc, j = p & (core - 1);
    int sum = 0;
    for (int k = 0; k < qsize; k++) sum += (int)M[(k << lc) + j] * (int)sc.tmp[k * 33 + i];
    int v = iclip((sum + add2) >> shift2, -32768, 32767);
    if (rep == 1) block[i * bpitch + j] = (int16_t)v;
    else
      for (int m = 0; m < rep; m++)
        for (int n = 0; n < rep; n++) block[(i * rep + m) * bpitch + j * rep + n] = (int16_t)v;
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------
// a12: quantize.  enc/encode_block.c:84-160.  coef: compact qsize x qsize (raster).  The level_mode hysteresis is a
// two-state machine along the zig-zag scan; each lane simulates its 8-position chunk for both start states, a warp
// scan composes the state maps, then each lane replays its chunk from the true start state.
// ---------------------------------------------------------------------------------------------------------------
__constant__ uint16_t c_quant[6] = {26214, 23302, 20560, 18396, 16384, 14564};  // common/common_tables.c:72
__constant__ uint16_t c_dequant[6] = {40, 45, 51, 57, 64, 72};                  // common/common_tables.c:73

// scan index of raster position (r,c) in an n x n zig-zag (common/common_tables.c:29-62), closed form
__device__ __forceinline__ int zigzag_index(int r, int c, int n) {
  int d = r + c;
  int before = d < n ? d * (d + 1) / 2 : n * n - (2 * n - 1 - d) * (2 * n - d) / 2;  // samples on earlier diagonals
  int lo = d < n ? 0 : d - (n - 1);  // smallest row index on this diagonal
  // odd diagonals run top-right -> bottom-left (row ascending), even ones the other way
  int k = (d & 1) ? (r - lo) : ((d < n ? d : n - 1) - r);
  return before + k;
}

// T = int when every intermediate fits 32 bits (scale <= 26214, |coef| <= 32768 -> product < 2^30; offsets <= 115 << (shift2 - 8)
// stay below 2^27 for shift2 <= 28), int64_t otherwise: same values, a third of the multiply instructions.
template <class T> __device__ __forceinline__ int warp_quantize_t(const int16_t *coef, int16_t *coefq, int qp, int size, int coeff_type, TxScratch &sc, int shift2, const uint8_t *zz16) {
  const int lane = lane_id();
  const int intra = (coeff_type >> 1) & 1, qsize = min(size, 16), nq = qsize * qsize, lq = ilog2(qsize);
  const T scale = c_quant[qp % 6];
  int *scan = (int *)sc.in;  // reuse: 256 ints of scan-ordered coefficients
  const bool tab = zz16 != nullptr && qsize == 16;  // 16x16 scan positions from a shared-memory table instead of the closed form
  for (int p = lane; p < nq; p += 32) scan[tab ? (int)zz16[p] : zigzag_index(p >> lq, p & (qsize - 1), qsize)] = coef[p];
  __syncwarp();
  // each lane owns `per` (<= 8) consecutive scan positions; their three candidate levels are computed ONCE and kept in registers:
  // level0 = ac >> shift2 decides between the two rounding offsets, lvA / lvB are the levels with off0 / off1
  const T unit = (T)1 << (shift2 - 8);
  const T off_last = (T)(intra ? 38 : -26) * unit;
  const T off0 = (T)(intra ? 102 : 51) * unit, off1 = (T)(intra ? 115 : 90) * unit;
  const int per = (nq + 31) / 32, p0 = lane * per;
  int cv[8], l0[8], lvA[8], lvB[8];
  int last = -1;
#pragma unroll
  for (int t = 0; t < 8; t++) {
    const int p = p0 + t;
    cv[t] = (t < per && p < nq) ? scan[p] : 0;
    const T ac = scale * (T)iabs(cv[t]);
    l0[t] = (int)(ac >> shift2);
    lvA[t] = (int)((ac + off0) >> shift2);
    lvB[t] = (int)((ac + off1) >> shift2);
    const T l = ac + off_last;
    if (t < per && p < nq && (int)((l > 0 ? l : -l) >> shift2)) last = p;  // last_pos: highest position whose level with the "last" offset is non-zero
  }
  last = (int)__reduce_max_sync(FULL, (unsigned)(last + 1)) - 1;
  unsigned map = 0;  // bit s = end state when the chunk is entered in state s
#pragma unroll
  for (int st = 0; st < 2; st++) {
    int mode = st;
#pragma unroll
    for (int t = 0; t < 8; t++) {
      if (t < per && p0 + t <= last) {
        const int level = (l0[t] > (1 - mode)) ? lvB[t] : lvA[t];
        if (mode) { if (level == 0) mode = 0; }
        else if (level > 1) mode = 1;
      }
    }
    map |= (unsigned)mode << st;
  }
  // inclusive scan of map composition: state after chunk L given state before chunk 0
  // compose(f then g)(s) = g(f(s)); represent as 2-bit maps
  unsigned incl = map;
  for (int o = 1; o < 32; o <<= 1) {
    unsigned prev = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) {
      unsigned r0 = (incl >> ((prev >> 0) & 1)) & 1, r1 = (incl >> ((prev >> 1) & 1)) & 1;
      incl = r0 | (r1 << 1);
    }
  }
  unsigned before = __shfl_up_sync(FULL, incl, 1);
  int mode = lane == 0 ? 1 : (int)((before >> 1) & 1);  // initial level_mode = 1
  int cbp = 0;
#pragma unroll
  for (int t = 0; t < 8; t++) {
    const int p = p0 + t;
    if (t < per && p < nq) {
      int q = 0;
      if (p <= last) {
        const int level = (l0[t] > (1 - mode)) ? lvB[t] : lvA[t];
        q = cv[t] < 0 ? -level : level;
        cbp |= level != 0;
        if (mode) { if (level == 0) mode = 0; }
        else if (level > 1) mode = 1;
      }
      sc.tmp[p] = (int16_t)q;  // scan order
    }
  }
  __syncwarp();
  for (int p = lane; p < nq; p += 32) coefq[p] = sc.tmp[tab ? (int)zz16[p] : zigzag_index(p >> lq, p & (qsize - 1), qsize)];
  __syncwarp();
  return __any_sync(FULL, cbp);
}
__device__ int warp_quantize(const int16_t *coef, int16_t *coefq, int qp, int size, int coeff_type, TxScratch &sc, const uint8_t *zz16 = nullptr) {
  const int shift2 = 21 - ilog2(size) + qp / 6;
  return shift2 <= 28 ? warp_quantize_t<int>(coef, coefq, qp, size, coeff_type, sc, shift2, zz16) : warp_quantize_t<int64_t>(coef, coefq, qp, size, coeff_type, sc, shift2, zz16);
}

// ---------------------------------------------------------------------------------------------------------------
// SURVEY 8f.2: bits that write_coeff() (enc/write_bits.c:145-242) emits for the quantised block, from the code lengths of
// put_vlc() (enc/putvlc.c:73-161).  The coder walks the zig-zag scan in two modes — level mode (every position coded,
// left by coding a zero) and run mode (zero runs + the next level; re-enters level mode after a level > 1) — so, like the
// quantiser's hysteresis, it is a two-state machine over the scan: state entering position p, the adaptive-table flag
// (level of position p - 1 if that was coded in level mode) and the run length (distance to the last coded position)
// are all prefix quantities.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int vlc_len(int n, unsigned cn) {  // tables 0, 1, 6, 10
  if (n == 10) return 1 + 2 * ilog2((int)cn + 1);
  if (n == 6) {
    if (!cn) return 2;
    cn++;
    n = 2;
  }
  if ((int)cn < (5 << n)) return 1 + n + (int)(cn >> n);
  return (5 - n) + 1 + 2 * ilog2((int)(cn - (5u << n) + (1u << n)));
}
struct CoeffBitCtx {
  int chroma, intra, run_tab;
  unsigned eob_pos;
  __device__ __forceinline__ CoeffBitCtx(int size, int type) : chroma(type & 1), intra((type >> 1) & 1), run_tab(((type & 1) && size <= 8) ? 10 : 6), eob_pos((type & 1) ? 0u : 2u) {}
  // bits of one position; S = mode entering it (1 level, 0 run), A = adaptive-table flag, run = zeros since the last coded position
  __device__ __forceinline__ int pos_bits(int c, int S, int A, int run) const {
    const int lev = iabs(c);
    if (S) return vlc_len(A, (unsigned)lev) + (lev > 0);
    if (!c) return 0;
    const unsigned cn = lev == 1 ? (unsigned)(run * 5) >> 2 : (unsigned)(run * 5 + 4);
    return vlc_len(run_tab, cn + (cn >= eob_pos)) + (lev > 1 ? vlc_len(0, (unsigned)((lev - 2) * 2 + (c < 0))) : 1);
  }
  __device__ __forceinline__ int tail_bits(int last, int N, int S_last, int c_last) const {  // after the last non-zero position
    const int lev = iabs(c_last), S_end = S_last ? 1 : lev > 1;
    const int A_end = (!chroma && S_last) ? lev > 3 : 0;
    int pos = last + 1, bits = 0;
    if (pos < N && S_end) { bits += vlc_len(A_end, 0); pos++; }
    if (pos < N) bits += vlc_len(run_tab, eob_pos);
    return bits;
  }
};
// one thread, N scan-ordered levels (registers when the loops unroll, local memory otherwise)
template <int N, class Q> __device__ __forceinline__ int thread_coeff_bits(const Q &q, int size, int type) {
  const CoeffBitCtx cx(size, type);
  int last = -1;
#pragma unroll(N <= 16 ? N : 1)
  for (int p = 0; p < N; p++)
    if (q[p]) last = p;
  if (last < 0) return 0;
  int bits = 0;
  if (cx.chroma) {
    if (last == 0 && iabs(q[0]) == 1) return 2;
    bits = 1;
  }
  int S = 1, A = cx.intra && !cx.chroma, ev = -1, S_last = 1;
#pragma unroll(N <= 16 ? N : 1)
  for (int p = 0; p < N; p++) {
    if (p <= last) {
      const int c = q[p], lev = iabs(c);
      bits += cx.pos_bits(c, S, A, p - 1 - ev);
      if (p == last) S_last = S;
      if (S) { if (!cx.chroma) A = lev > 3; if (!lev) S = 0; ev = p; }
      else if (c) { S = lev > 1; ev = p; }
    }
  }
  return bits + cx.tail_bits(last, N, S_last, q[last]);
}
// whole warp, nq (<= 256) scan-ordered levels in shared memory; every lane returns the total
__device__ int warp_coeff_bits(const int16_t *scan, int nq, int size, int type) {
  const CoeffBitCtx cx(size, type);
  const int lane = lane_id(), per = (nq + 31) >> 5, p0 = lane * per;
  int mylast = -1;
  for (int t = 0; t < per; t++)
    if (p0 + t < nq && scan[p0 + t]) mylast = p0 + t;
  const int last = (int)__reduce_max_sync(FULL, (unsigned)(mylast + 1)) - 1;
  if (last < 0) return 0;
  int bits = 0;
  if (cx.chroma) {
    if (last == 0 && iabs(scan[0]) == 1) return 2;
    bits = lane == 0 ? 1 : 0;
  }
  // state map of the chunk for both entry states, composed across lanes (see warp_quantize_t)
  unsigned map = 0;
  for (int st = 0; st < 2; st++) {
    int S = st;
    for (int t = 0; t < per; t++) {
      const int p = p0 + t;
      if (p > last) break;
      const int lev = iabs(scan[p]);
      S = S ? lev != 0 : lev > 1;
    }
    map |= (unsigned)S << st;
  }
  unsigned incl = map;
  for (int o = 1; o < 32; o <<= 1) {
    unsigned prev = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) {
      unsigned r0 = (incl >> ((prev >> 0) & 1)) & 1, r1 = (incl >> ((prev >> 1) & 1)) & 1;
      incl = r0 | (r1 << 1);
    }
  }
  const unsigned before = __shfl_up_sync(FULL, incl, 1);
  const int S0 = lane == 0 ? 1 : (int)((before >> 1) & 1);  // the scan starts in level mode
  // first walk: state entering the chunk's last position and the chunk's last coded position
  int S = S0, Sin_last = S0, ev = -1;
  for (int t = 0; t < per; t++) {
    const int p = p0 + t;
    if (p > last) break;
    const int lev = iabs(scan[p]);
    Sin_last = S;
    if (S || lev) ev = p;
    S = S ? lev != 0 : lev > 1;
  }
  // previous lane's last position: its entry state and level (for the adaptive flag); exclusive prefix maximum of ev
  const int pS = __shfl_up_sync(FULL, Sin_last, 1), pc = lane ? (int)scan[p0 - 1] : 0;
  int evx = ev;
  for (int o = 1; o < 32; o <<= 1) {
    int v = __shfl_up_sync(FULL, evx, o);
    if (lane >= o) evx = max(evx, v);
  }
  int evprev = __shfl_up_sync(FULL, evx, 1);
  if (lane == 0) evprev = -1;
  // second walk: bits
  S = S0;
  int A = lane == 0 ? (cx.intra && !cx.chroma) : ((!cx.chroma && pS) ? iabs(pc) > 3 : 0);
  ev = evprev;
  for (int t = 0; t < per; t++) {
    const int p = p0 + t;
    if (p > last) break;
    const int c = scan[p], lev = iabs(c);
    bits += cx.pos_bits(c, S, A, p - 1 - ev);
    if (p == last) bits += cx.tail_bits(last, nq, S, c);
    if (S) { A = cx.chroma ? 0 : lev > 3; if (!lev) S = 0; ev = p; }
    else if (c) { S = lev > 1; ev = p; A = 0; }
  }
  return (int)warp_sum((uint32_t)bits);
}

// ---------------------------------------------------------------------------------------------------------------
// 4x4 transform blocks (68 % of all transform blocks in the HDB mix): ONE THREAD runs the whole chain
// residual -> 4-point DCT x2 -> quantize -> dequantize -> inverse DCT x2 -> reconstruct -> SSD in registers.
// Same arithmetic as the generic routines (common/transform.c:281-307, 411-465 with the 4x4 matrix :63-68,
// enc/encode_block.c:84-160, common/common_block.c:45-83); the butterflies are exact integer refactorings of the
// matrix products.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dct4_fwd(int a0, int a1, int a2, int a3, int &y0, int &y1, int &y2, int &y3) {
  int e0 = a0 + a3, e1 = a1 + a2, o0 = a0 - a3, o1 = a1 - a2;
  y0 = 64 * (e0 + e1); y2 = 64 * (e0 - e1); y1 = 83 * o0 + 36 * o1; y3 = 36 * o0 - 83 * o1;
}
__device__ __forceinline__ void dct4_inv(int x0, int x1, int x2, int x3, int &y0, int &y1, int &y2, int &y3) {
  int e0 = 64 * (x0 + x2), e1 = 64 * (x0 - x2), o0 = 83 * x1 + 36 * x3, o1 = 36 * x1 - 83 * x3;
  y0 = e0 + o0; y1 = e1 + o1; y2 = e1 - o1; y3 = e0 - o0;
}
template <class S> __device__ __forceinline__ void load_row4(const S *p, int (&v)[4]) {
  if (sizeof(S) == 1) {
    uint32_t w = ldw_any(p);
#pragma unroll
    for (int i = 0; i < 4; i++) v[i] = (int)((w >> (8 * i)) & 0xff);
  } else {
    uint32_t w0 = ldw_any(p), w1 = ldw_any(p + 2);
    v[0] = (int)(w0 & 0xffff); v[1] = (int)(w0 >> 16); v[2] = (int)(w1 & 0xffff); v[3] = (int)(w1 >> 16);
  }
}
template <class S> __device__ __forceinline__ void store_row4(S *p, const int (&v)[4]) {
  if (sizeof(S) == 1 && (((uintptr_t)p) & 3) == 0) {
    *(uint32_t *)p = (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24);
  } else if (sizeof(S) == 2 && (((uintptr_t)p) & 3) == 0) {
    ((uint32_t *)p)[0] = (uint32_t)v[0] | ((uint32_t)v[1] << 16);
    ((uint32_t *)p)[1] = (uint32_t)v[2] | ((uint32_t)v[3] << 16);
  } else {
#pragma unroll
    for (int i = 0; i < 4; i++) p[i] = (S)v[i];
  }
}

// returns cbp; ssd out
template <class S>
__device__ int thread_txfm4(const S *orig, int os, const S *pred, int ps, S *rec, int rs, int16_t *coeffq_out, int qp, int coeff_type, int bitdepth,
                            uint64_t &ssd_out, int want_bits, int &bits_out) {
  constexpr int ZZ[16] = {0, 1, 5, 6, 2, 4, 7, 12, 3, 8, 11, 13, 9, 10, 14, 15};  // raster -> scan (common/common_tables.c:29-34)
  const int maxv = (1 << bitdepth) - 1;
  int o[16], p[16], t[16], c[16];
#pragma unroll
  for (int r = 0; r < 4; r++) {
    int a[4], b[4];
    load_row4<S>(orig + r * os, a);
    load_row4<S>(pred + r * ps, b);
#pragma unroll
    for (int k = 0; k < 4; k++) { o[r * 4 + k] = a[k]; p[r * 4 + k] = b[k]; }
  }
  // forward, 1st dimension: t[i][j] = (sum_k M[i][k] * res[j][k] + add1) >> shift1 (int16)
  const int shift1 = bitdepth - 6, add1 = 1 << (shift1 - 1);
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int y0, y1, y2, y3;
    dct4_fwd(o[j * 4] - p[j * 4], o[j * 4 + 1] - p[j * 4 + 1], o[j * 4 + 2] - p[j * 4 + 2], o[j * 4 + 3] - p[j * 4 + 3], y0, y1, y2, y3);
    t[0 * 4 + j] = (int16_t)((y0 + add1) >> shift1); t[1 * 4 + j] = (int16_t)((y1 + add1) >> shift1);
    t[2 * 4 + j] = (int16_t)((y2 + add1) >> shift1); t[3 * 4 + j] = (int16_t)((y3 + add1) >> shift1);
  }
  // 2nd dimension: coef[i][j] = (sum_k M[i][k] * t[j][k] + 64) >> 7, stored straight into scan order
  int sc[16];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int y0, y1, y2, y3;
    dct4_fwd(t[j * 4], t[j * 4 + 1], t[j * 4 + 2], t[j * 4 + 3], y0, y1, y2, y3);
    sc[ZZ[0 * 4 + j]] = (int16_t)((y0 + 64) >> 7); sc[ZZ[1 * 4 + j]] = (int16_t)((y1 + 64) >> 7);
    sc[ZZ[2 * 4 + j]] = (int16_t)((y2 + 64) >> 7); sc[ZZ[3 * 4 + j]] = (int16_t)((y3 + 64) >> 7);
  }
  // quantize (enc/encode_block.c:84-160), size 4: shift2 = 19 + qp/6; products fit 32 bits (|c| * 26214 + offset < 2^31)
  const int intra = (coeff_type >> 1) & 1, scale = c_quant[qp % 6], shift2 = 19 + qp / 6;
  const int off_last = (intra ? 38 : -26) * (1 << (shift2 - 8));
  int last = -1;
#pragma unroll
  for (int pos = 0; pos < 16; pos++) {
    int l = iabs(sc[pos]) * scale + off_last;
    if ((iabs(l) >> shift2) != 0) last = pos;
  }
  const int off0 = (intra ? 102 : 51) << (shift2 - 8), off1 = (intra ? 115 : 90) << (shift2 - 8);
  int mode = 1, cbp = 0, q[16];
#pragma unroll
  for (int pos = 0; pos < 16; pos++) {
    int lev = 0;
    if (pos <= last) {
      int ac = scale * iabs(sc[pos]);
      int level0 = ac >> shift2;
      lev = (ac + ((level0 > (1 - mode)) ? off1 : off0)) >> shift2;
      cbp |= lev != 0;
      if (mode) { if (lev == 0) mode = 0; }
      else if (lev > 1) mode = 1;
    }
    q[pos] = sc[pos] < 0 ? -lev : lev;
  }
  if (coeffq_out) {
#pragma unroll
    for (int r = 0; r < 16; r++) coeffq_out[r] = (int16_t)q[ZZ[r]];
  }
  bits_out = (want_bits && cbp) ? thread_coeff_bits<16>(q, 4, coeff_type) : 0;
  uint64_t ssd = 0;
  if (cbp) {
    // dequantize (common/common_block.c:45-73), size 4: rshift = 1
    const int lshift = qp / 6, dscale = c_dequant[qp % 6];
#pragma unroll
    for (int r = 0; r < 16; r++) {
      int v = q[ZZ[r]] * dscale;
      c[r] = lshift >= 1 ? (int)(int16_t)((unsigned)v << (lshift - 1)) : (int)(int16_t)((v + 1) >> 1);
    }
    // inverse, 1st dimension: t[i][j] = clip16((sum_k M[k][j] * c[k][i] + 64) >> 7)
#pragma unroll
    for (int i = 0; i < 4; i++) {
      int y0, y1, y2, y3;
      dct4_inv(c[0 * 4 + i], c[1 * 4 + i], c[2 * 4 + i], c[3 * 4 + i], y0, y1, y2, y3);
      t[i * 4 + 0] = iclip((y0 + 64) >> 7, -32768, 32767); t[i * 4 + 1] = iclip((y1 + 64) >> 7, -32768, 32767);
      t[i * 4 + 2] = iclip((y2 + 64) >> 7, -32768, 32767); t[i * 4 + 3] = iclip((y3 + 64) >> 7, -32768, 32767);
    }
    // 2nd dimension + reconstruction: out[i][j] = clip16((sum_k M[k][j] * t[k][i] + add2) >> (20 - bitdepth))
    const int shiftB = 20 - bitdepth, addB = 1 << (shiftB - 1);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      int y[4];
      dct4_inv(t[0 * 4 + i], t[1 * 4 + i], t[2 * 4 + i], t[3 * 4 + i], y[0], y[1], y[2], y[3]);
      int v[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        int r = iclip((y[j] + addB) >> shiftB, -32768, 32767);
        v[j] = sat_px(r + p[i * 4 + j], maxv);
        int d = o[i * 4 + j] - v[j];
        ssd += (uint32_t)(d * d);
      }
      if (rec) store_row4<S>(rec + i * rs, v);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; i++) {
      int v[4];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        v[j] = p[i * 4 + j];
        int d = o[i * 4 + j] - v[j];
        ssd += (uint32_t)(d * d);
      }
      if (rec) store_row4<S>(rec + i * rs, v);
    }
  }
  ssd_out = ssd;
  return cbp;
}

// 8x8 transform blocks: also one THREAD per block.  The 64-entry work arrays live in local memory, which the hardware
// interleaves per thread, so the lock-step (uniform-index) accesses of a warp coalesce into L1 lines; the DCT matrix is
// read from the shared-memory table with a warp-uniform index (broadcast).  Same arithmetic as warp_fwd_transform /
// warp_quantize / warp_dequantize / warp_inv_transform.
__constant__ uint8_t c_zz8[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30, 41, 43, 9,  11, 18, 24, 31, 40, 44, 53,
                                   10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};
// eight-term dot product of an int8 matrix row (two words) with eight int16 values (four words): four DP2A
__device__ __forceinline__ int dot8(uint2 m, uint4 v, int acc) {
  acc = __dp2a_lo((int)v.x, (int)m.x, acc);
  acc = __dp2a_hi((int)v.y, (int)m.x, acc);
  acc = __dp2a_lo((int)v.z, (int)m.y, acc);
  return __dp2a_hi((int)v.w, (int)m.y, acc);
}
template <class S>
__device__ int thread_txfm8(const S *orig, int os, const S *pred, int ps, S *rec, int rs, int16_t *coeffq_out, int qp, int coeff_type, int bitdepth,
                            const int8_t *tab8, const int8_t *tab8t, uint64_t &ssd_out, int want_bits, int &bits_out) {
  const uint2 *M = (const uint2 *)(tab8 + dct_tab8_ofs(3)), *Mt = (const uint2 *)(tab8t + dct_tab8_ofs(3));  // rows of 8 int8, warp-uniform index
  const int maxv = (1 << bitdepth) - 1;
  alignas(16) int16_t a[64], b[64];  // 16-byte rows: each row is one 128-bit local load in the matrix phases
  for (int r = 0; r < 8; r++) {
    int o0[4], o1[4], p0[4], p1[4];
    load_row4<S>(orig + r * os, o0); load_row4<S>(orig + r * os + 4, o1);
    load_row4<S>(pred + r * ps, p0); load_row4<S>(pred + r * ps + 4, p1);
    *(uint4 *)&a[r * 8] = make_uint4(((uint32_t)(o0[0] - p0[0]) & 0xffffu) | ((uint32_t)(o0[1] - p0[1]) << 16), ((uint32_t)(o0[2] - p0[2]) & 0xffffu) | ((uint32_t)(o0[3] - p0[3]) << 16),
                                     ((uint32_t)(o1[0] - p1[0]) & 0xffffu) | ((uint32_t)(o1[1] - p1[1]) << 16), ((uint32_t)(o1[2] - p1[2]) & 0xffffu) | ((uint32_t)(o1[3] - p1[3]) << 16));
  }
  // forward: b[i][j] = (M[i] . res[j] + add1) >> shift1, then a[scan(i, j)] = (M[i] . b[j] + 128) >> 8
  const int shift1 = 3 + bitdepth - 8, add1 = 1 << (shift1 - 1);
  for (int j = 0; j < 8; j++) {
    const uint4 v = *(const uint4 *)&a[j * 8];
#pragma unroll
    for (int i = 0; i < 8; i++) b[i * 8 + j] = (int16_t)(dot8(M[i], v, add1) >> shift1);
  }
  for (int j = 0; j < 8; j++) {
    const uint4 v = *(const uint4 *)&b[j * 8];
#pragma unroll
    for (int i = 0; i < 8; i++) a[c_zz8[i * 8 + j]] = (int16_t)(dot8(M[i], v, 128) >> 8);  // scan order
  }
  const int intra = (coeff_type >> 1) & 1, scale = c_quant[qp % 6], shift2 = 18 + qp / 6;
  const int off_last = (intra ? 38 : -26) * (1 << (shift2 - 8));
  int last = -1;
  for (int pos = 0; pos < 64; pos++) {
    int l = iabs((int)a[pos]) * scale + off_last;
    if ((iabs(l) >> shift2) != 0) last = pos;
  }
  const int off0 = (intra ? 102 : 51) << (shift2 - 8), off1 = (intra ? 115 : 90) << (shift2 - 8);
  int mode = 1, cbp = 0;
  for (int pos = 0; pos < 64; pos++) {
    int lev = 0, cc = a[pos];
    if (pos <= last) {
      int ac = scale * iabs(cc);
      int level0 = ac >> shift2;
      lev = (ac + ((level0 > (1 - mode)) ? off1 : off0)) >> shift2;
      cbp |= lev != 0;
      if (mode) { if (lev == 0) mode = 0; }
      else if (lev > 1) mode = 1;
    }
    b[pos] = (int16_t)(cc < 0 ? -lev : lev);  // quantised, scan order
  }
  if (coeffq_out)
    for (int p = 0; p < 64; p++) coeffq_out[p] = b[c_zz8[p]];
  bits_out = (want_bits && cbp) ? thread_coeff_bits<64>(b, 8, coeff_type) : 0;
  uint64_t ssd = 0;
  if (cbp) {
    // de-quantise into the TRANSPOSED block a[i][k] = rcoeff[k][i], so that both inverse stages are row . row products
    const int lshift = qp / 6, dscale = c_dequant[qp % 6];  // rshift = 2
    for (int k = 0; k < 8; k++)
#pragma unroll
      for (int i = 0; i < 8; i++) {
        int v = (int)b[c_zz8[k * 8 + i]] * dscale;
        a[i * 8 + k] = lshift >= 2 ? (int16_t)((unsigned)v << (lshift - 2)) : (int16_t)((v + (1 << (1 - lshift))) >> (2 - lshift));
      }
    // inverse 1st dimension: T[i][j] = clip16((sum_k M[k][j] * rcoeff[k][i] + 64) >> 7), stored transposed: b[j][i]
    for (int i = 0; i < 8; i++) {
      const uint4 v = *(const uint4 *)&a[i * 8];
#pragma unroll
      for (int j = 0; j < 8; j++) b[j * 8 + i] = (int16_t)iclip(dot8(Mt[j], v, 64) >> 7, -32768, 32767);
    }
    // 2nd dimension + reconstruction: out[i][j] = clip16((sum_k M[k][j] * T[k][i] + addB) >> shiftB) = Mt[j] . b[i]
    const int shiftB = 20 - bitdepth, addB = 1 << (shiftB - 1);
    for (int i = 0; i < 8; i++) {
      const uint4 v = *(const uint4 *)&b[i * 8];
#pragma unroll
      for (int h2 = 0; h2 < 2; h2++) {
        int pv[4], ov[4], o4[4];
        load_row4<S>(pred + i * ps + 4 * h2, pv);
        load_row4<S>(orig + i * os + 4 * h2, ov);
#pragma unroll
        for (int t = 0; t < 4; t++) {
          int r = iclip(dot8(Mt[4 * h2 + t], v, addB) >> shiftB, -32768, 32767);
          o4[t] = sat_px(r + pv[t], maxv);
          int d = ov[t] - o4[t];
          ssd += (uint32_t)(d * d);
        }
        if (rec) store_row4<S>(rec + i * rs + 4 * h2, o4);
      }
    }
  } else {
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int h2 = 0; h2 < 2; h2++) {
        int pv[4], ov[4];
        load_row4<S>(pred + i * ps + 4 * h2, pv);
        load_row4<S>(orig + i * os + 4 * h2, ov);
        if (rec) store_row4<S>(rec + i * rs + 4 * h2, pv);
#pragma unroll
        for (int t = 0; t < 4; t++) { int d = ov[t] - pv[t]; ssd += (uint32_t)(d * d); }
      }
  }
  ssd_out = ssd;
  return cbp;
}

// a13: dequantize.  common/common_block.c:45-73 (no weight matrix).  compact in, compact out (pitch qsize)
__device__ void warp_dequantize(const int16_t *cq, int16_t *rc, int qp, int size) {
  const int lshift = qp / 6, qsize = min(size, 16), rshift = ilog2(size) - 1;
  const int64_t scale = c_dequant[qp % 6];
  const int64_t add = lshift < rshift ? (1 << (rshift - lshift - 1)) : 0;
  for (int p = lane_id(); p < qsize * qsize; p += 32) {
    int c = cq[p];
    rc[p] = lshift >= rshift ? (int16_t)((c * scale) << (lshift - rshift)) : (int16_t)((c * scale + add) >> (rshift - lshift));
  }
  __syncwarp();
}

// a14: calc_cbp_simd semantics.  enc/enc_kernels.c:828-909 (int16 column sums; 4x4: odd + |even| per pair)
__device__ int warp_calc_cbp(const int16_t *block, int size, int thr) {
  const int lane = lane_id();
  int hit = 0;
  int16_t col = 0;
  if (lane < size)
    for (int i = 0; i < size; i++) col = (int16_t)(col + block[i * size + lane]);
  int16_t a = (int16_t)(col < 0 ? -col : col);
  if (size == 4) {
    int odd = __shfl_down_sync(FULL, (int)col, 1);
    if (lane < 4 && !(lane & 1)) hit = (odd + (int)a) > thr;
  } else if (lane < size)
    hit = a > (int16_t)thr;
  return __any_sync(FULL, hit);
}

// common/common_kernels.c:127-161
__device__ int warp_check_nz_area(const int16_t *coeff, int size) {
  const int qs = min(size, 16), lq = ilog2(qs);
  int ndc = 0, n4 = 0, n8 = 0;
  for (int p = lane_id(); p < qs * qs; p += 32) {
    int i = p >> lq, j = p & (qs - 1);
    if (coeff[i * size + j]) {
      if (i || j) ndc = 1;
      if (i >= 4 || j >= 4) n4 = 1;
      if (i >= 8 || j >= 8) n8 = 1;
    }
  }
  ndc = __any_sync(FULL, ndc);
  n4 = __any_sync(FULL, n4);
  n8 = __any_sync(FULL, n8);
  if (size == 4) return ndc ? 3 : 0;
  if (size == 8) return !ndc ? 0 : (!n4 ? 1 : 2);
  return !ndc ? 0 : (!n4 ? 1 : (!n8 ? 2 : 3));
}

// ---------------------------------------------------------------------------------------------------------------
// a15: intra prediction.  common/intra_prediction.c:57-428.  left/top hold 2*size samples (shared memory).
// ---------------------------------------------------------------------------------------------------------------
template <class S>
__device__ void warp_make_top_and_left(S *left, S *top, S &top_left, const S *rec_frame, int fstride, const S *rblock, int rbstride, int i, int j,
                                       int ypos, int xpos, int size, int cb_upright, int cb_downleft, int tb_split, int bitdepth) {
  const int lane = lane_id();
  const S mid = (S)(128 << (bitdepth - 8));
  int downleft, upright;
  if (!tb_split) { downleft = cb_downleft; upright = cb_upright; }
  else {
    downleft = (j == 0 && (i == 0 || cb_downleft)) ? 1 : 0;
    upright = (j == 0 || (i == 0 && cb_upright)) ? 1 : 0;
  }
  const int leftlen = downleft ? size + 1 : size, toplen = upright ? size + 1 : size;
  S tl = mid;
  if (ypos + i == 0) {
    TB_ROLL
    for (int k = lane; k < 2 * size; k += 32) top[k] = mid;
  } else {
    const S *src = (i == 0) ? rec_frame - fstride + j : rblock - rbstride;
    S val = TB_LDF(src + toplen - 1);
    TB_ROLL
    for (int k = lane; k < 2 * size; k += 32) top[k] = k < toplen ? TB_LDF(src + k) : (k >= size ? val : TB_LDF(src + k));
    if (xpos > 0) tl = (i == 0) ? TB_LDF(rec_frame - fstride + j - 1) : ((j > 0) ? TB_LDF(rblock - rbstride - 1) : TB_LDF(rec_frame + (i - 1) * fstride - 1));
    else tl = TB_LDF(src);
  }
  if (xpos + j == 0) {
    TB_ROLL
    for (int k = lane; k < 2 * size; k += 32) left[k] = mid;
  } else {
    const S *base = (j == 0) ? rec_frame + i * fstride - 1 : rblock - 1;
    const int st = (j == 0) ? fstride : rbstride;
    S val = TB_LDF(base + (leftlen - 1) * st);
    TB_ROLL
    for (int k = lane; k < 2 * size; k += 32) left[k] = k < leftlen ? TB_LDF(base + k * st) : (k >= size ? val : TB_LDF(base + k * st));
  }
  __syncwarp();
  if (ypos + i == 0) tl = left[0];
  top_left = tl;
}

template <class S> __device__ __forceinline__ int f121(const S *in, int k, int len) {
  int a = in[k > 0 ? k - 1 : 0], b = in[k], c = in[k < len - 1 ? k + 1 : len - 1];
  return (a + 2 * b + c + 2) >> 2;
}
template <class S> __device__ __forceinline__ int f12221(const S *in, int k, int len) {  // planar pre-filter, int16 in the reference
  int a = in[max(k - 2, 0)], b = in[max(k - 1, 0)], c = in[min(k + 1, len - 1)], d = in[min(k + 2, len - 1)];
  return (int)(int16_t)(a + 2 * b + 2 * in[k] + 2 * c + d);
}

// filt: scratch of 4*size+1 samples for the 1-2-1 filtered arrays
template <class S>
__device__ void warp_intra_pred(const S *left, const S *top, S top_left, int ypos, int xpos, int size, S *pblock, int pstride, int mode, int bitdepth,
                                S *filt) {
  const int lane = lane_id(), ls = ilog2(size), maxv = (1 << bitdepth) - 1;
  if (mode < 0 || mode > 9) mode = 0;
  S *tF = filt, *lF = filt + 2 * size;
  int tlF = 0, dc = 0;
  int16_t ptlF = 0;
  if (mode == 4 || mode == 7 || mode == 8) {
    TB_ROLL
    for (int k = lane; k < size; k += 32) { tF[k] = (S)f121<S>(top, k, size); lF[k] = (S)f121<S>(left, k, size); }
    tlF = (int)(S)((2 * (int)top_left + left[0] + top[0] + 2) >> 2);
  } else if (mode == 5 || mode == 6) {
    TB_ROLL
    for (int k = lane; k < 2 * size; k += 32) tF[k] = (S)f121<S>(top, k, 2 * size);
  } else if (mode == 9) {
    TB_ROLL
    for (int k = lane; k < 2 * size; k += 32) lF[k] = (S)f121<S>(left, k, 2 * size);
  } else if (mode == 0) {
    const S *l = xpos != 0 ? left : top, *t = ypos != 0 ? top : left;
    unsigned sum = 0;
    TB_ROLL
    for (int k = lane; k < size; k += 32) sum += (unsigned)t[k] + (unsigned)l[k];
    sum = warp_sum(sum);
    dc = (int)((sum + (unsigned)size) / (2u * (unsigned)size));
  } else if (mode == 1) {
    ptlF = (int16_t)(left[1] + 2 * left[0] + 2 * (int)top_left + 2 * top[0] + top[1]);
  }
  __syncwarp();
  TB_ROLL
  for (int p = lane; p < size * size; p += 32) {
    int i = p >> ls, j = p & (size - 1), v, d;
    switch (mode) {
      case 0: v = dc; break;
      case 1: v = sat_px((f12221<S>(left, i, size) + f12221<S>(top, j, size) - ptlF + 4) / 8, maxv); break;
      case 2: v = left[i]; break;
      case 3: v = top[j]; break;
      case 4: d = i - j; v = d > 0 ? lF[d - 1] : (d == 0 ? tlF : tF[-d - 1]); break;
      case 5: v = tF[i + j + 1]; break;
      case 6: d = i + 2 * j; v = (d & 1) ? tF[(d + 1) / 2] : (tF[d / 2] + tF[d / 2 + 1]) >> 1; break;
      case 7:
        d = i - 2 * j;
        if (d > 1) v = lF[d - 2];
        else if (d == 1) v = tlF;
        else if (d == 0) v = (tlF + tF[0]) >> 1;
        else v = (d & 1) ? tF[(-d) / 2] : (tF[(-d) / 2] + tF[(-d) / 2 - 1]) >> 1;
        break;
      case 8:
        d = 2 * i - j;
        if (d < -1) v = tF[-d - 2];
        else if (d == -1) v = tlF;
        else if (d == 0) v = (tlF + lF[0]) >> 1;
        else v = (d & 1) ? lF[d / 2] : (lF[d / 2] + lF[d / 2 - 1]) >> 1;
        break;
      default: d = 2 * i + j; v = (d & 1) ? lF[(d + 1) / 2] : (lF[d / 2] + lF[d / 2 + 1]) >> 1; break;
    }
    pblock[i * pstride + j] = (S)v;
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------
// a16: chroma-from-luma.  common/common_block.c:347-427 (4:2:0, sub = 1)
// ---------------------------------------------------------------------------------------------------------------
template <class S> __device__ void warp_cfl(const S *y, S *u, S *v, const S *ry, int n, int cstride, int stride, int sub, int bitdepth) {
  const int lane = lane_id(), nc = n >> sub, lognc = ilog2(nc), cs = cstride >> sub, maxv = (1 << bitdepth) - 1, ln = ilog2(n);
  int64_t sq = 0;
  TB_ROLL
  for (int p = lane; p < n * n; p += 32) {
    int i = p >> ln, j = p & (n - 1);
    int d = (int)ry[i * stride + j] - (int)y[i * n + j];
    sq += d * d;
  }
  sq = (int64_t)warp_sum64((uint64_t)sq);
  if ((sq >> (2 * ln)) <= (64 << 2 * (bitdepth - 8))) return;
  int64_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // ysum usum vsum yy yu yv uu vv
  TB_ROLL
  for (int p = lane; p < nc * nc; p += 32) {
    int i = p >> lognc, j = p & (nc - 1);
    int us = u[i * cs + j], vs = v[i * cs + j];
    int ys = sub ? ((int)y[(2 * i) * n + 2 * j] + y[(2 * i) * n + 2 * j + 1] + y[(2 * i + 1) * n + 2 * j] + y[(2 * i + 1) * n + 2 * j + 1] + 2) >> 2
                 : (int)y[i * cstride + j];
    acc[0] += ys; acc[1] += us; acc[2] += vs;
    acc[3] += ys * ys; acc[4] += ys * us; acc[5] += ys * vs; acc[6] += us * us; acc[7] += vs * vs;
  }
#pragma unroll
  for (int k = 0; k < 8; k++) acc[k] = (int64_t)warp_sum64((uint64_t)acc[k]);
  const int sh = lognc * 2;
  int64_t ysum = acc[0], usum = acc[1], vsum = acc[2];
  int64_t ssyy = acc[3] - (ysum * ysum >> sh), ssuu = acc[6] - (usum * usum >> sh), ssvv = acc[7] - (vsum * vsum >> sh);
  int64_t ssyu = acc[4] - (ysum * usum >> sh), ssyv = acc[5] - (ysum * vsum >> sh);
  if (!ssyy) return;
  for (int c = 0; c < 2; c++) {
    int64_t sc = c ? ssyv : ssyu, scc = c ? ssvv : ssuu, csum = c ? vsum : usum;
    S *dst = c ? v : u;
    if (!(sc * sc * 2 > ssyy * scc)) continue;
    int64_t a64 = (sc << 16) / ssyy;
    int64_t b64 = ((csum << 16) - a64 * ysum) >> sh;
    int64_t lim = (int64_t)1 << (31 - bitdepth);
    int32_t a = (int32_t)(a64 < -lim ? -lim : (a64 > lim ? lim : a64));
    int64_t bb = b64 + (1 << 15);
    int64_t lo = -((int64_t)1 << 31), hi = ((int64_t)1 << 31) - 1;
    int32_t b = (int32_t)(bb < lo ? lo : (bb > hi ? hi : bb));
    TB_ROLL
    for (int p = lane; p < nc * nc; p += 32) {
      int i = p >> lognc, j = p & (nc - 1);
      int out;
      if (sub) {
        const S *r0 = ry + (2 * i) * stride + 2 * j, *r1 = r0 + stride;
        out = (sat_px((a * (int)r0[0] + b) >> 16, maxv) + sat_px((a * (int)r0[1] + b) >> 16, maxv) + sat_px((a * (int)r1[0] + b) >> 16, maxv) +
               sat_px((a * (int)r1[1] + b) >> 16, maxv) + 2) >> 2;
      } else
        out = sat_px((a * (int)ry[i * stride + j] + b) >> 16, maxv);
      dst[i * cs + j] = (S)out;
    }
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------------
// a18/a19 scalar pieces.  common/common_block.c:214-220, 315-321; common/common_frame.h:61-65
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int constrain(int diff, int threshold, unsigned damping) {
  if (!threshold) return 0;
  int a = iabs(diff);
  int lim = max(0, threshold - (a >> (damping - (unsigned)ilog2(threshold))));
  lim = min(a, lim);
  return diff < 0 ? -lim : lim;
}
__device__ __forceinline__ int clpf_sample(int X, int A, int B, int C, int D, int E, int F, int G, int H, int s, unsigned dmp) {
  int delta = constrain(A - X, s, dmp) + 3 * constrain(B - X, s, dmp) + constrain(C - X, s, dmp) + 3 * constrain(D - X, s, dmp) +
              3 * constrain(E - X, s, dmp) + constrain(F - X, s, dmp) + 3 * constrain(G - X, s, dmp) + constrain(H - X, s, dmp);
  return (8 + delta - (delta < 0)) >> 4;
}
__device__ __forceinline__ int adjust_strength(int strength, int var) {
  int i = (var >> 6) ? min(ilog2(var >> 6), 12) : 0;
  return var ? (strength * (4 + i) + 8) >> 4 : 0;
}
__constant__ int8_t c_cdef_dx[8][2] = {{1, 2}, {1, 2}, {1, 2}, {1, 2}, {1, 2}, {0, 1}, {0, 0}, {0, -1}};   // common/common_block.c:189-208
__constant__ int8_t c_cdef_dy[8][2] = {{-1, -2}, {0, -1}, {0, 0}, {0, 1}, {1, 2}, {1, 2}, {1, 2}, {1, 2}};

// One CDEF output sample from a uint16 staging tile `in` (pitch ss, 30000 = outside the frame).
// common/common_block.c:224-281 (CDEF_FULL = 0)
__device__ __forceinline__ int cdef_sample(const uint16_t *in, int ss, int pri_strength, int sec_strength, int dir, int pri_damping, int sec_damping,
                                           int coeff_shift) {
  const int sel = (pri_strength >> coeff_shift) & 1;
  const int pt0 = sel ? 3 : 4, pt1 = sel ? 3 : 2, st0 = 2, st1 = 1;
  int x = (int16_t)in[0], mx = x, mn = x, sum = 0;
#pragma unroll
  for (int k = 0; k < 2; k++) {
    int o0 = c_cdef_dy[dir][k] * ss + c_cdef_dx[dir][k];
    int o1 = c_cdef_dy[(dir + 2) & 7][k] * ss + c_cdef_dx[(dir + 2) & 7][k];
    int o2 = c_cdef_dy[(dir + 6) & 7][k] * ss + c_cdef_dx[(dir + 6) & 7][k];
    int pt = k ? pt1 : pt0, st = k ? st1 : st0;
    int p[2] = {(int16_t)in[o0], (int16_t)in[-o0]};
    int s4[4] = {(int16_t)in[o1], (int16_t)in[-o1], (int16_t)in[o2], (int16_t)in[-o2]};
#pragma unroll
    for (int t = 0; t < 2; t++) {
      sum += pt * constrain(p[t] - x, pri_strength, (unsigned)pri_damping);
      if (p[t] != 30000) mx = max(mx, p[t]);
      mn = min(mn, p[t]);
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
      sum += st * constrain(s4[t] - x, sec_strength, (unsigned)sec_damping);
      if (s4[t] != 30000) mx = max(mx, s4[t]);
      mn = min(mn, s4[t]);
    }
  }
  sum = (int)(int16_t)sum;
  int y = x + ((8 + sum - (sum < 0)) >> 4);
  return iclip(y, mn, mx);
}

// CDEF direction search on an 8x8 block, one warp.  common/common_block.c:94-167.  Returns dir; *var out.
template <class S> __device__ int warp_cdef_find_dir(const S *img, int stride, int coeff_shift, int &var_out) {
  // Each lane owns one or more line sums.  partial[d][n]: 8 directions x up to 15 lines = 120 sums -> 4 per lane.
  const int lane = lane_id();
  // load the block into registers: lane l holds pixels (row l>>2, cols (l&3)*2, +1) -> 64 pixels over 32 lanes
  int r = lane >> 2, c0 = (lane & 3) * 2;
  int x0 = ((int)img[r * stride + c0] >> coeff_shift) - 128, x1 = ((int)img[r * stride + c0 + 1] >> coeff_shift) - 128;
  // cost accumulation: every lane computes complete line sums by gathering pixels through shuffles would be
  // shuffle-heavy; the block is only 64 samples, so each lane instead recomputes the line sums it owns from the
  // two-sample registers of all lanes via 32 shuffles.
  int32_t cost_part[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const int div_table[9] = {0, 840, 420, 280, 210, 168, 140, 120, 105};
  // lane L < 15 owns line index L of every direction
  int sums[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int src = 0; src < 32; src++) {
    int a = __shfl_sync(FULL, x0, src), b = __shfl_sync(FULL, x1, src);
    int i = src >> 2, j = (src & 3) * 2;
#pragma unroll
    for (int t = 0; t < 2; t++) {
      int x = t ? b : a, jj = j + t;
      if (i + jj == lane) sums[0] += x;
      if (i + jj / 2 == lane) sums[1] += x;
      if (i == lane) sums[2] += x;
      if (3 + i - jj / 2 == lane) sums[3] += x;
      if (7 + i - jj == lane) sums[4] += x;
      if (3 - i / 2 + jj == lane) sums[5] += x;
      if (jj == lane) sums[6] += x;
      if (i / 2 + jj == lane) sums[7] += x;
    }
  }
  // weights per line index for each direction class
  if (lane < 15) {
    int w045 = lane < 7 ? div_table[lane + 1] : (lane == 7 ? div_table[8] : div_table[15 - lane]);  // dirs 0 and 4: 15 lines
    cost_part[0] = sums[0] * sums[0] * w045;
    cost_part[4] = sums[4] * sums[4] * w045;
    if (lane < 8) {
      cost_part[2] = sums[2] * sums[2] * div_table[8];
      cost_part[6] = sums[6] * sums[6] * div_table[8];
    }
    if (lane < 11) {
      // odd directions: 11 lines; lines 3..7 weight div[8], lines j and 10-j (j<3) weight div[2j+2]
      int wodd = (lane >= 3 && lane <= 7) ? div_table[8] : (lane < 3 ? div_table[2 * lane + 2] : div_table[2 * (10 - lane) + 2]);
      cost_part[1] = sums[1] * sums[1] * wodd;
      cost_part[3] = sums[3] * sums[3] * wodd;
      cost_part[5] = sums[5] * sums[5] * wodd;
      cost_part[7] = sums[7] * sums[7] * wodd;
    }
  }
  int32_t cost[8];
#pragma unroll
  for (int d = 0; d < 8; d++) cost[d] = (int32_t)warp_sum((uint32_t)cost_part[d]);
  int32_t best_cost = 0;
  int best_dir = 0;
#pragma unroll
  for (int d = 0; d < 8; d++)
    if (cost[d] > best_cost) { best_cost = cost[d]; best_dir = d; }
  int32_t orth = 0;
#pragma unroll
  for (int d = 0; d < 8; d++)
    if (d == ((best_dir + 4) & 7)) orth = cost[d];
  var_out = (best_cost - orth) >> 10;
  return best_dir;
}

}  // namespace tb
