// tb_rdo.h — the reference's per-super-block RD loop (SURVEY.md §8f.1, §8f.2), written once for two builds:
//   * nvcc, device backend (tb_rdo.cu): the product — one 8-warp CTA per super block at a time inside the persistent rdo_batch_kernel;
//   * g++,  oracle backend (oracle/rdo_hostcheck.cpp): TEST INFRASTRUCTURE — the same control flow over the plain-C oracle's
//     primitives, used here (no GPU in the build container) to pin the control flow against the compiled reference SB by SB.
// The control flow is scalar and warp-uniform, and it is SPMD over the NW warps of a CTA (NW = 1 on the host unless the host check
// simulates warps with threads): every warp executes the whole control flow on its own scratch blocks (Work), so sequential sections
// (neighbour derivation, the bipred refinement, the recursion itself) are simply replicated and stay consistent without communication.
// Two kinds of sections are DISTRIBUTED: the motion searches of the reference frames (one reference per warp; results exchanged through
// the backend and the candidate lists replayed by the other warps) and the RD candidates of a block (round robin in the serial form of the
// decision, drawn from shared counters in the overlapped form: mode_decision_overlap).  The reference keeps the first candidate with the
// strictly smallest cost; that is the minimum of (cost, k), k = the candidate's position in the reference's evaluation order, which the
// backend's reduction returns together with the warp that holds the winning reconstruction; that warp alone commits the block.
// The backend's primitives are the warp-cooperative routines of tb_device.cuh.  Nothing in this file touches samples directly.
//
// What is restated (reference file:line at each function): process_block enc/encode_block.c:2401-2565, early skip :2123-2399,
// mode_decision_rdo :1835-2120, search_{intra,inter,bipred}_prediction_params :928-1098, 1679-1833, encode_block :1340-1514 with
// encode_and_reconstruct_block_{intra,intra_uv,inter} :1100-1338, cost_calc :916, copy_best_parameters :1615, copy_deblock_data
// :1568, add_mvcandidate :71; the bit counts of write_super_mode / write_block / write_mv / write_delta_qp enc/write_bits.c:122-600
// with put_vlc enc/putvlc.c:73-161; get_mv_pred / get_mv_merge / get_mv_skip common/inter_prediction.c:413-836,
// get_inter_prediction_yuv :185-233, average_blocks_all :235-256; find_block_contexts common/common_block.c:283-303;
// get_{up,left,upright,downleft}_available common/common_block.h:52-95.
// Not restated (tb_rdo_encode_frame rejects these settings): sync, qmtx, interp_ref == 2, delta QP / rate control, 4:4:4 / 4:0:0.
#pragma once
#include <stdint.h>
#include "../../include/thor_b200.h"

// TBR_NI: the functions of the control flow exist ONCE in the device code (no inlining at their many call sites): the RD loop is one kernel whose warps run
// different parts of it at the same time, and an all-inlined build (2.5 MB of SASS) lives on instruction fetches from L2
#ifdef __CUDACC__
#define TBR_NI __noinline__
#else
#define TBR_NI
#endif
#ifdef __CUDACC__
#define TBR_HD __device__  // under nvcc the header is only instantiated for the device backend
#else
#define TBR_HD
#endif

namespace tbr {

enum { MODE_SKIP = 0, MODE_INTRA, MODE_INTER, MODE_BIPRED, MODE_MERGE };
enum { PART_NONE = 0, PART_HOR, PART_VER, PART_QUAD };
enum { I_FRAME = 0, P_FRAME, B_FRAME };
enum { MIN_BLOCK = 8, MIN_PB = 4, MAX_TR = 128, EARLY_SKIP_BLOCK = 32 };
// phases of one block decision for the device's timers (be.mark(k): the time since the previous mark belongs to phase k)
enum { PH_OTHER = 0, PH_EARLY_SKIP, PH_SKIP_MERGE, PH_SEARCH, PH_INTER_CAND, PH_BIPRED, PH_INTRA_SEARCH, PH_INTRA_CAND, PH_COMMIT, PH_N };
constexpr uint32_t MAX_U32 = 1u << 31;  // MAX_UINT32 of common/global.h:62 (sic: 1<<31)

typedef tb_mv_t Mv;
struct IPred { Mv mv0, mv1; int ref_idx0, ref_idx1, bipred_flag; };  // inter_pred_t
struct Ctx3 { int split, cbp, index; };                               // block_context_t

TBR_HD inline int imin(int a, int b) { return a < b ? a : b; }
TBR_HD inline int imax(int a, int b) { return a > b ? a : b; }
TBR_HD inline int iabs_(int a) { return a < 0 ? -a : a; }
// tb_rdo_coeff_count of thor_b200.h for both builds
TBR_HD inline int coeff_count(int size, int tb_split) { const int t = tb_split ? size / 2 : size, q = t < 16 ? t : 16; return (tb_split ? 4 : 1) * q * q; }
TBR_HD inline int ilog2_(unsigned x) { int r = 0; while (x >>= 1) r++; return r; }

// lambda * n + 0.5 without FMA contraction (the reference is ISO C on x86-64: separate multiply and add)
TBR_HD inline double mul_add_half(double lambda, double n) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(__dmul_rn(lambda, n), 0.5);
#else
  volatile double m = lambda * n;
  return m + 0.5;
#endif
}

// put_vlc code lengths, enc/putvlc.c:73-161
TBR_HD inline int vlc_len(int n, unsigned cn) {
  const unsigned e = 5;
  if (n < 0) return -n;
  if (n == 6 || n == 7) {
    if (!cn) return 2;
    if (n == 6) { cn++; n = 2; }
    else {
      if (cn == 1) return 3;
      if (cn < 4) return 4;
      cn += 4; n = 3;
    }
  }
  if (n <= 5) {
    if ((int)cn < (int)(e * (1u << n))) return 1 + n + (int)(cn >> n);
    unsigned code = cn - (e * (1u << n)) + (1u << n);
    return (int)(e - n) + 1 + 2 * ilog2_(code);
  }
  if (n == 8) return cn < 6 ? 2 + (int)(cn >> 1) : 5;
  if (n == 10) return 1 + 2 * ilog2_(cn + 1);
  return cn == (unsigned)(n - 10) ? n - 10 : (int)cn + 1;  // 11..18
}
// write_mv, enc/write_bits.c:122-143 (the difference is taken in int16 like mv_t)
TBR_HD inline int mv_bits(Mv mv, Mv mvp) {
  int16_t dx = (int16_t)(mv.x - mvp.x), dy = (int16_t)(mv.y - mvp.y);
  unsigned ax = (uint16_t)iabs_(dx), ay = (uint16_t)iabs_(dy);
  return vlc_len(7, ax) + (ax > 0) + vlc_len(7, ay) + (ay > 0);
}

// common/common_block.h:52-95
TBR_HD inline int upright_available(int ypos, int xpos, int bw, int bh, int fw, int /*fh*/, int sb) {
  int a = (ypos > 0) && (xpos + bw < fw);
  int size = imax(bw, bh);
  for (int s2 = size; s2 < sb; s2 *= 2)
    if ((ypos % (s2 << 1)) == s2 && (xpos % s2) == (s2 - size)) a = 0;
  return a;
}
TBR_HD inline int downleft_available(int ypos, int xpos, int bw, int bh, int /*fw*/, int fh, int sb) {
  int a = (xpos > 0) && (ypos + bh < fh);
  int size = imax(bw, bh);
  if ((ypos % sb) == (sb - size) && (xpos % sb) == 0) a = 0;
  for (int s2 = 2 * size; s2 <= sb; s2 *= 2)
    if ((ypos % s2) == (s2 - size) && (xpos % s2) > 0) a = 0;
  return a;
}

// frame-level state the RD loop reads and writes (pointers are in the address space of the build: host or device)
template <class S> struct FrameCtx {
  int width, height, sb_size, bitdepth, frame_type, qp, qpc, num_ref, interp_ref, num_intra_modes;
  double lambda, sqrt_lambda;
  int enable_bipred, enable_tb_split, enable_pb_split, speed, intra_rdo, use_block_contexts, cfl_intra, cfl_inter;
  float early_skip_thr;
  int ref_sign[TB_RDO_MAX_REF], ref_sign_ge[TB_RDO_MAX_REF];
  const S *org[3]; int org_stride[2];
  const S *ref[TB_RDO_MAX_REF][3]; int ref_stride[2];
  S *rec[3]; int rec_stride[2];
  tb_rdo_blk_t *blk; int blk_stride;
  tb_rdo_leaf_t *leaves; int *leaf_count; int16_t *coeffs;
};

// block_param_t without the coefficient arrays (those live in Work)
struct Cand {
  int mode, intra_mode, skip_idx, pb_part;
  Mv mv0[4], mv1[4];
  int ref_idx0, ref_idx1, dir;
  int cbp_y, cbp_u, cbp_v;
  int tb_param, tb_split;
};
// one transform chain of a candidate (residual -> DCT -> quant -> dequant -> inverse DCT -> reconstruction): the chains of a candidate's planes and
// transform blocks are independent of each other when the predictions are complete, so the backend may run them side by side (tx_multi)
template <class S> struct TxJob {
  const S *orig; const S *pred; S *rec; int16_t *cq;
  int os, ps, rs, size, qp, coeff_type, fast;
};
// block_info_t
struct BlockInfo {
  int size, ypos, xpos, bwidth, bheight;
  IPred skip_cand[2], merge_cand[2];
  int num_skip, num_merge;
  Mv mvp;
  int max_tb, max_pb;
  Ctx3 ctx;
  Cand best;  // block_info->block_param
};

// per-super-block scratch (global memory on the device): compact blocks with pitch = size like the reference's yuv_block_t
template <class S> struct Work {
  S rec_y[128 * 128], rec_u[64 * 64], rec_v[64 * 64];     // rec_block: the candidate being evaluated
  S best_y[128 * 128], best_u[64 * 64], best_v[64 * 64];  // rec_block_best
  S p_y[128 * 128], p_u[64 * 64], p_v[64 * 64];           // pblock
  S p0_y[128 * 128], p0_u[64 * 64], p0_v[64 * 64];        // pblock0
  S p1_y[128 * 128], p1_u[64 * 64], p1_v[64 * 64];        // pblock1
  S org8[128 * 128];
  int16_t cq_y[1024], cq_u[1024], cq_v[1024];             // candidate coefficients (reference layout: transform block k at k*256)
  int16_t bq_y[1024], bq_u[1024], bq_v[1024];             // best
  // top-down (encoder_speed > 0, 16x16): the parent's best survives its children's evaluation
  S td_y[16 * 16], td_u[8 * 8], td_v[8 * 8];
  int16_t tdq_y[1024], tdq_u[1024], tdq_v[1024];
  Mv mvcand[TB_RDO_MAX_REF][64];                          // frame_info->mvcand: reset per super block (enc/encode_frame.c:702-705)
  int mvcand_num[TB_RDO_MAX_REF];
  uint64_t mvcand_mask[TB_RDO_MAX_REF];
};

template <class S, class B> struct Rdo {
  FrameCtx<S> &F;
  Work<S> &W;    // this warp's scratch
  Work<S> &W0;   // warp 0's scratch: holds the CTA-shared top-down save area
  B &be;
  int best_ref;      // frame_info->best_ref (per super block)
  int sb_index;
  int n_leaves, coeff_used;
  // distributed candidate evaluation: running candidate index and this warp's best so far
  int cidx, loc_idx;
  uint32_t loc_cost, loc_worst, loc_bestc;
  // the candidate about to be evaluated has the same inter prediction as the previous one of this warp (same vectors, another tb_param): W.p_* is still valid
  bool reuse_pred;

  TBR_HD Rdo(FrameCtx<S> &f, Work<S> &w, Work<S> &w0, B &b)
      : F(f), W(w), W0(w0), be(b), best_ref(-1), sb_index(0), n_leaves(0), coeff_used(0), cidx(0), loc_idx(0), loc_cost(MAX_U32), loc_worst(0), loc_bestc(MAX_U32), reuse_pred(false) {}

  // ---------------------------------------------------------------------------------------------------------------
  // neighbour state
  // ---------------------------------------------------------------------------------------------------------------
  TBR_HD IPred ipred_at(int index) const {
    const tb_rdo_blk_t b = be.ld_blk(F.blk + index);  // another CTA may have written it: the device backend bypasses L1
    IPred p; p.mv0 = b.mv0; p.mv1 = b.mv1; p.ref_idx0 = b.ref_idx0; p.ref_idx1 = b.ref_idx1; p.bipred_flag = b.bipred_flag;
    return p;
  }
  TBR_HD static IPred zero_pred() { IPred p; p.mv0.x = p.mv0.y = p.mv1.x = p.mv1.y = 0; p.ref_idx0 = p.ref_idx1 = 0; p.bipred_flag = 0; return p; }

  // common/inter_prediction.c:413-524
  TBR_HD TBR_NI Mv get_mv_pred(int ypos, int xpos, int bw, int bh) const {
    const int size = imax(bw, bh), bsz = size / MIN_PB, bst = F.blk_stride, bi = (ypos / MIN_PB) * bst + xpos / MIN_PB;
    const int up0 = bi - bst, up1 = bi - bst + (bsz - 1) / 2, up2 = bi - bst + bsz - 1, l0 = bi - 1, l1 = bi + bst * ((bsz - 1) / 2) - 1,
              l2 = bi + bst * (bsz - 1) - 1, dl = bi + bst * bsz - 1, ur = bi - bst + bsz, ul = bi - bst - 1;
    const int U = ypos > 0, L = xpos > 0, UR = upright_available(ypos, xpos, bw, bh, F.width, F.height, F.sb_size),
              DL = downleft_available(ypos, xpos, bw, bh, F.width, F.height, F.sb_size);
    int a = -1, b = -1, c = -1;
    if (U == 0 && UR == 0 && L == 0 && DL == 0) {}
    else if (U == 1 && UR == 0 && L == 0 && DL == 0) { a = up0; b = up1; c = up2; }
    else if (U == 1 && UR == 1 && L == 0 && DL == 0) { a = up0; b = up2; c = ur; }
    else if (U == 0 && UR == 0 && L == 1 && DL == 0) { a = l0; b = l1; c = l2; }
    else if (U == 1 && UR == 0 && L == 1 && DL == 0) { a = ul; b = up2; c = l2; }
    else if (U == 1 && UR == 1 && L == 1 && DL == 0) { a = up0; b = ur; c = l2; }
    else if (U == 0 && UR == 0 && L == 1 && DL == 1) { a = l0; b = l2; c = dl; }
    else if (U == 1 && UR == 0 && L == 1 && DL == 1) { a = up2; b = l0; c = dl; }
    else if (U == 1 && UR == 1 && L == 1 && DL == 1) { a = up0; b = ur; c = l0; }
    Mv z; z.x = z.y = 0;
    const Mv mva = a >= 0 ? be.ld_blk(F.blk + a).mv0 : z, mvb = b >= 0 ? be.ld_blk(F.blk + b).mv0 : z, mvc = c >= 0 ? be.ld_blk(F.blk + c).mv0 : z;
    Mv p;
    p.x = (int16_t)(mva.x < mvb.x ? imin(mvb.x, imax(mva.x, mvc.x)) : imin(mva.x, imax(mvb.x, mvc.x)));
    p.y = (int16_t)(mva.y < mvb.y ? imin(mvb.y, imax(mva.y, mvc.y)) : imin(mva.y, imax(mvb.y, mvc.y)));
    return p;
  }
  // get_mv_merge / get_mv_skip (LIMITED_SKIP = 1: two candidates, identical derivation), common/inter_prediction.c:526-836
  TBR_HD TBR_NI int get_mv_skip_merge(int ypos, int xpos, int bw, int bh, IPred *out) const {
    const int size = imax(bw, bh), bsz = size / MIN_PB, bst = F.blk_stride, bi = (ypos / MIN_PB) * bst + xpos / MIN_PB;
    const int up0 = bi - bst, l0 = bi - 1, ur = bi - bst + bsz;
    int up2 = bi - bst + bsz - 1, l2 = bi + bst * (bsz - 1) - 1;
    const int U = ypos > 0, L = xpos > 0, UR = upright_available(ypos, xpos, bw, bh, F.width, F.height, F.sb_size);
    if (ypos + size > F.height) l2 = l0;
    if (xpos + size > F.width) up2 = up0;
    IPred t[2];
    t[0] = L ? ipred_at(l2) : zero_pred();
    t[1] = UR ? ipred_at(ur) : (U ? ipred_at(up2) : zero_pred());
    out[0] = t[0];
    int n = 1;
    const bool dup = t[1].mv0.x == out[0].mv0.x && t[1].mv0.y == out[0].mv0.y && t[1].ref_idx0 == out[0].ref_idx0 && t[1].mv1.x == out[0].mv1.x &&
                     t[1].mv1.y == out[0].mv1.y && t[1].ref_idx1 == out[0].ref_idx1 && (t[1].bipred_flag == out[0].bipred_flag || t[1].bipred_flag == -1);
    if (!dup) out[n++] = t[1];
    return n;
  }
  // common/common_block.c:283-303
  TBR_HD TBR_NI Ctx3 find_block_contexts(int ypos, int xpos, int size) const {
    Ctx3 c;
    if (ypos >= MIN_BLOCK && xpos >= MIN_BLOCK && ypos + size < F.height && xpos + size < F.width && F.use_block_contexts && size <= MAX_TR) {
      const int bs = F.blk_stride, bi = (ypos / MIN_PB) * bs + xpos / MIN_PB;
      const tb_rdo_blk_t u = be.ld_blk(F.blk + bi - bs), l = be.ld_blk(F.blk + bi - 1);
      c.split = (u.size < size) + (l.size < size);
      c.cbp = (u.cbp_y > 0) + (l.cbp_y > 0);
      c.index = 3 * c.split + ((u.cbp_y > 0 || u.cbp_u > 0 || u.cbp_v > 0) + (l.cbp_y > 0 || l.cbp_u > 0 || l.cbp_v > 0));
    } else c.split = c.cbp = c.index = -1;
    return c;
  }
  // enc/encode_block.c:69-82
  TBR_HD void add_mvcandidate(Mv mv, int ref_idx) {
    Mv imv; imv.x = (int16_t)((mv.x + 2) >> 2); imv.y = (int16_t)((mv.y + 2) >> 2);
    const uint64_t m = (uint64_t)1 << (((imv.y << 3) ^ imv.x) & 63);
    if (!(m & W.mvcand_mask[ref_idx])) { W.mvcand[ref_idx][W.mvcand_num[ref_idx]] = imv; W.mvcand_num[ref_idx] += 1; }
    W.mvcand_mask[ref_idx] |= m;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // bits: write_super_mode + write_block, enc/write_bits.c:255-600 (counting only)
  // ---------------------------------------------------------------------------------------------------------------
  TBR_HD TBR_NI int super_mode_bits(const BlockInfo &bi, const Cand &c, int split_flag, int encode_this_size) const {
    const int size = bi.size;
    if (F.frame_type != I_FRAME) {
      if (!encode_this_size) return 1;
      int code = 0;
      const int bipred_possible = F.num_ref > 1 && F.enable_bipred, split_possible = size > MIN_BLOCK;
      int maxbit = 2 + F.num_ref + split_possible + bipred_possible;
      if (F.interp_ref > 2) maxbit -= 1;
      const bool ctx_swap = bi.ctx.index == 2 || bi.ctx.index > 3;
      if (split_flag == 1) {
        if (size > MAX_TR) return 1;
        code = 1;
        if (ctx_swap) code = (code + 3) % 4;
        return vlc_len(10 + maxbit, code);
      }
      const int mode = c.mode;
      if (F.interp_ref) {
        if (mode == MODE_SKIP) code = 0;
        else if (mode == MODE_MERGE) code = 2;
        else if (mode == MODE_BIPRED) code = 3;
        else if (mode == MODE_INTRA) code = 4;
        else if (mode == MODE_INTER && c.ref_idx0 > 0) code = 4 + c.ref_idx0;
        else code = 4 + F.num_ref;
        if (!bipred_possible && code > 3) code -= 1;
        if (!split_possible && code > 1) code -= 1;
        if (ctx_swap && size > MIN_BLOCK && code < 3) code = (code + 2) % 3;
      } else {
        if (mode == MODE_SKIP) code = 0;
        else if (mode == MODE_INTER && c.ref_idx0 == 0) code = 2;
        else if (mode == MODE_MERGE) code = 3;
        else if (mode == MODE_BIPRED) code = 4;
        else if (mode == MODE_INTRA) code = 5;
        else if (mode == MODE_INTER && c.ref_idx0 > 0) code = 5 + c.ref_idx0;
        if (!bipred_possible && code > 4) code -= 1;
        if (!split_possible && code > 1) code -= 1;
        if (ctx_swap && size > MIN_BLOCK && code < 4) code = (code + 3) % 4;
      }
      return vlc_len(10 + maxbit, code);
    }
    return (encode_this_size && (size > MIN_BLOCK || split_flag == 1)) ? 1 : 0;
  }

  TBR_HD int coeff_bits_plane(const int16_t *cq, int size, int type) const { return be.coeff_bits(cq, size, type); }

  TBR_HD TBR_NI int block_bits(const BlockInfo &bi, const Cand &c, const int16_t *cqy, const int16_t *cqu, const int16_t *cqv) const {
    const int size = bi.size, tb_split = c.tb_split, mode = c.mode, size_uv = size >> 1;
    const int coeff_type = (mode == MODE_INTRA) << 1;
    static const int8_t cbp_table_[8] = {1, 0, 5, 2, 6, 3, 7, 4};
    int cbp_y = c.cbp_y & 255, cbp_u = c.cbp_u & 255, cbp_v = c.cbp_v & 255;
    const int encode_this_size = bi.ypos + size <= F.height && bi.xpos + size <= F.width;
    int bits = super_mode_bits(bi, c, 0, encode_this_size);
    if (mode == MODE_INTRA) bits += F.num_intra_modes <= 4 ? 2 : vlc_len(8, c.intra_mode);
    else if (mode == MODE_INTER) {
      if (bi.max_pb > 1) bits += vlc_len(13, c.pb_part);
      Mv mvp2 = bi.mvp;
      bits += mv_bits(c.mv0[0], mvp2);
      if (c.pb_part == PART_HOR) { mvp2 = c.mv0[0]; bits += mv_bits(c.mv0[2], mvp2); }
      else if (c.pb_part == PART_VER) { mvp2 = c.mv0[0]; bits += mv_bits(c.mv0[1], mvp2); }
      else if (c.pb_part == PART_QUAD) { mvp2 = c.mv0[0]; bits += mv_bits(c.mv0[1], mvp2) + mv_bits(c.mv0[2], mvp2) + mv_bits(c.mv0[3], mvp2); }
    } else if (mode == MODE_BIPRED) {
      Mv mvp2 = bi.mvp;
      if (c.pb_part == PART_NONE) bits += mv_bits(c.mv0[0], mvp2);
      if (F.frame_type == B_FRAME) mvp2 = c.mv0[0];
      bits += mv_bits(c.mv1[0], mvp2);
      if (c.pb_part == PART_HOR) { mvp2 = c.mv1[0]; bits += mv_bits(c.mv1[2], mvp2); }
      else if (c.pb_part == PART_VER) { mvp2 = c.mv1[0]; bits += mv_bits(c.mv1[1], mvp2); }
      else if (c.pb_part == PART_QUAD) { mvp2 = c.mv1[0]; bits += mv_bits(c.mv1[1], mvp2) + mv_bits(c.mv1[2], mvp2) + mv_bits(c.mv1[3], mvp2); }
      if (F.frame_type == P_FRAME) bits += F.num_ref == 2 ? vlc_len(13, 2 * c.ref_idx0 + c.ref_idx1) : vlc_len(10, 4 * c.ref_idx0 + c.ref_idx1);
    } else if (mode == MODE_SKIP || mode == MODE_MERGE) {
      const int nvec = mode == MODE_SKIP ? bi.num_skip : bi.num_merge;
      if (nvec == 4) bits += 2;
      else if (nvec == 3) bits += vlc_len(12, c.skip_idx);
      else if (nvec == 2) bits += 1;
    }
    if (mode != MODE_SKIP) {
      const int max_tb = bi.max_tb;
      int code;
      const int off = mode == MODE_MERGE ? 1 : 2;
      if (max_tb > 1 && tb_split) code = off;
      else {
        const int cbp = cbp_y + (cbp_u << 1) + (cbp_v << 2);
        code = cbp_table_[cbp];
        if (mode == MODE_MERGE) { if (code == 1) code = 7; else if (code > 1) code -= 1; }
        else if (bi.ctx.cbp == 0 && code < 2) code = 1 - code;
        if (max_tb > 1 && code >= off) code++;
      }
      bits += vlc_len(0, code);
      if (tb_split == 0) {
        if (cbp_y) bits += coeff_bits_plane(cqy, size, coeff_type | 0);
        if (cbp_u) bits += coeff_bits_plane(cqu, size_uv, coeff_type | 1);
        if (cbp_v) bits += coeff_bits_plane(cqv, size_uv, coeff_type | 1);
      } else if (size_uv > 4) {
        for (int index = 0; index < 4; index++) {
          const int y = (c.cbp_y >> (3 - index)) & 1, u = (c.cbp_u >> (3 - index)) & 1, v = (c.cbp_v >> (3 - index)) & 1;
          int code2 = cbp_table_[y + (u << 1) + (v << 2)];
          if (bi.ctx.cbp == 0 && code2 < 2) code2 = 1 - code2;
          bits += vlc_len(0, code2);
          if (y) bits += coeff_bits_plane(cqy + index * 256, size / 2, coeff_type | 0);
          if (u) bits += coeff_bits_plane(cqu + index * 256, size_uv / 2, coeff_type | 1);
          if (v) bits += coeff_bits_plane(cqv + index * 256, size_uv / 2, coeff_type | 1);
        }
      } else {
        for (int index = 0; index < 4; index++) {
          const int y = (c.cbp_y >> (3 - index)) & 1;
          bits += 1;
          if (y) bits += coeff_bits_plane(cqy + index * 256, size / 2, coeff_type | 0);
        }
        // sic: cbp_u / cbp_v keep their whole-block values here (write_bits.c:583-590)
        bits += vlc_len(13, cbp_u + 2 * cbp_v);
        if (cbp_u) bits += coeff_bits_plane(cqu, size_uv, coeff_type | 1);
        if (cbp_v) bits += coeff_bits_plane(cqv, size_uv, coeff_type | 1);
      }
    }
    return bits;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // prediction
  // ---------------------------------------------------------------------------------------------------------------
  // get_inter_prediction_yuv, common/inter_prediction.c:185-233: pitch of the compact blocks = pos_size (block_pos->size)
  // luma_only: search_bipred_prediction_params (:1768) predicts all three planes but reads only the luma block; the chroma predictions have no effect
  TBR_HD TBR_NI void inter_pred_yuv(int ref_idx, S *py, S *pu, S *pv, int ypos, int xpos, int pos_size, int pbw, int pbh, const Mv *mv_arr, int sign, int split, int luma_only = 0) {
    const int div = split + 1, bw = pbw / div, bh = pbh / div, pst = pos_size, rsy = F.ref_stride[0], rsc = F.ref_stride[1];
    const int yc = ypos >> 1, xc = xpos >> 1;
    const S *ry = F.ref[ref_idx][0] + ypos * rsy + xpos, *ru = F.ref[ref_idx][1] + yc * rsc + xc, *rv = F.ref[ref_idx][2] + yc * rsc + xc;
    for (int index = 0; index < div * div; index++) {
      const int idx = index & 1, idy = (index >> 1) & 1;
      const int opy = idy * bh * pst + idx * bw, opc = (idy * bh * pst >> 2) + (idx * bw >> 1);
      const int ory = idy * bh * rsy + idx * bw, orc = (idy * bh * rsc >> 1) + (idx * bw >> 1);
      Mv mv = mv_arr[index];
      be.clip_mv(mv, ypos, xpos, F.width, F.height, bw, bh, sign);
      be.interp_luma(py + opy, pst, ry + ory, rsy, bw, bh, mv, sign, F.enable_bipred, F.width, F.height, xpos, ypos);
      if (luma_only) continue;
      be.interp_chroma(pu + opc, pst >> 1, ru + orc, rsc, bw >> 1, bh >> 1, mv, sign, F.width >> 1, F.height >> 1, xc, yc);
      be.interp_chroma(pv + opc, pst >> 1, rv + orc, rsc, bw >> 1, bh >> 1, mv, sign, F.width >> 1, F.height >> 1, xc, yc);
    }
  }
  // the inter prediction of a candidate into W.p_* (encode_block :1424-1451)
  TBR_HD TBR_NI void predict_inter(const BlockInfo &bi, const Cand &c) {
    const int split = (c.mode == MODE_INTER || c.mode == MODE_BIPRED) ? F.enable_pb_split : 0;
    if (c.dir == 2 || c.mode == MODE_BIPRED) {
      inter_pred_yuv(c.ref_idx0, W.p0_y, W.p0_u, W.p0_v, bi.ypos, bi.xpos, bi.size, bi.bwidth, bi.bheight, c.mv0, F.ref_sign[c.ref_idx0], split);
      inter_pred_yuv(c.ref_idx1, W.p1_y, W.p1_u, W.p1_v, bi.ypos, bi.xpos, bi.size, bi.bwidth, bi.bheight, c.mv1, F.ref_sign[c.ref_idx1], split);
      be.avg(W.p_y, W.p0_y, W.p1_y, bi.size, bi.bwidth, bi.bheight);
      be.avg(W.p_u, W.p0_u, W.p1_u, bi.size >> 1, bi.bwidth >> 1, bi.bheight >> 1);
      be.avg(W.p_v, W.p0_v, W.p1_v, bi.size >> 1, bi.bwidth >> 1, bi.bheight >> 1);
    } else
      inter_pred_yuv(c.ref_idx0, W.p_y, W.p_u, W.p_v, bi.ypos, bi.xpos, bi.size, bi.bwidth, bi.bheight, c.mv0, F.ref_sign[c.ref_idx0], split);
  }

  // encode_and_reconstruct_block_inter :1275-1338 for one plane (orig/pred/rec compact or strided; coefficients in the reference layout)
  TBR_HD TBR_NI int enc_rec_inter(const S *orig, int os, int size, int qp, const S *pred, int16_t *cq, S *rec, int coeff_type, int tb_split) {
    if (tb_split) {
      const int s2 = size / 2;
      int cbp = 0, index = 0;
      for (int i = 0; i < size; i += s2)
        for (int j = 0; j < size; j += s2) {
          const int fast = (size == 64 || F.speed > 1) ? 1 : 0;
          const int bit = be.tx_chain(orig + i * os + j, os, pred + i * size + j, size, rec + i * size + j, size, cq + index, s2, qp, coeff_type, fast);
          cbp = (cbp << 1) + bit;
          index += 256;
        }
      return cbp;
    }
    const int fast = ((size == 64 && F.speed > 0) || F.speed > 1) ? 1 : 0;
    return be.tx_chain(orig, os, pred, size, rec, size, cq, size, qp, coeff_type, fast);
  }
  // the chains of enc_rec_inter for one plane, appended to a job list (same order, same fast flags); returns the number of chains
  TBR_HD int inter_jobs(TxJob<S> *jobs, const S *orig, int os, int size, int qp, const S *pred, int16_t *cq, S *rec, int coeff_type, int tb_split) const {
    if (tb_split) {
      const int s2 = size / 2;
      int n = 0;
      for (int i = 0; i < size; i += s2)
        for (int j = 0; j < size; j += s2) {
          TxJob<S> &q = jobs[n];
          q.orig = orig + i * os + j; q.os = os; q.pred = pred + i * size + j; q.ps = size; q.rec = rec + i * size + j; q.rs = size; q.cq = cq + 256 * n; q.size = s2; q.qp = qp;
          q.coeff_type = coeff_type; q.fast = (size == 64 || F.speed > 1) ? 1 : 0;
          n++;
        }
      return 4;
    }
    TxJob<S> &q = jobs[0];
    q.orig = orig; q.os = os; q.pred = pred; q.ps = size; q.rec = rec; q.rs = size; q.cq = cq; q.size = size; q.qp = qp; q.coeff_type = coeff_type;
    q.fast = ((size == 64 && F.speed > 0) || F.speed > 1) ? 1 : 0;
    return 1;
  }
  TBR_HD static int join_cbp(const int *bit, int n) {
    int cbp = 0;
    for (int k = 0; k < n; k++) cbp = (cbp << 1) + bit[k];
    return cbp;
  }
  // encode_and_reconstruct_block_intra :1100-1168 (luma) — prediction into pblock (pitch size), reconstruction into rec_block (pitch size)
  TBR_HD TBR_NI int enc_rec_intra(const S *orig, int os, S *recf, int rfs, int ypos, int xpos, int size, int qp, S *pblock, int16_t *cq, S *rec_block, int coeff_type,
                           int tb_split, int intra_mode, int upright, int downleft) {
    const int fast = F.speed > 1;
    if (tb_split) {
      const int s2 = size / 2;
      int cbp = 0, index = 0;
      for (int i = 0; i < size; i += s2)
        for (int j = 0; j < size; j += s2) {
          be.intra_predict(pblock + i * size + j, size, recf, rfs, rec_block + i * size + j, size, i, j, ypos, xpos, s2, upright, downleft, 1, intra_mode);
          const int bit = be.tx_chain(orig + i * os + j, os, pblock + i * size + j, size, rec_block + i * size + j, size, cq + index, s2, qp, coeff_type, fast);
          cbp = (cbp << 1) + bit;
          index += 256;
        }
      return cbp;
    }
    be.intra_predict(pblock, size, recf, rfs, (const S *)nullptr, 0, 0, 0, ypos, xpos, size, upright, downleft, 0, intra_mode);
    return be.tx_chain(orig, os, pblock, size, rec_block, size, cq, size, qp, coeff_type, fast);
  }
  // the U and the V chain of one transform block: independent, side by side when they are thread-sized (<= 8x8)
  TBR_HD TBR_NI void uv_chains(const S *ou, const S *ov, int os, const S *pu, const S *pv, int ps, S *ru, S *rv, int rs, int16_t *cqu, int16_t *cqv, int size, int qp, int coeff_type,
                        int fast, int *bu, int *bv) {
    if (size <= 8) {
      TxJob<S> jobs[2];
      int bit[2];
      jobs[0].orig = ou; jobs[0].pred = pu; jobs[0].rec = ru; jobs[0].cq = cqu; jobs[1].orig = ov; jobs[1].pred = pv; jobs[1].rec = rv; jobs[1].cq = cqv;
      for (int k = 0; k < 2; k++) { jobs[k].os = os; jobs[k].ps = ps; jobs[k].rs = rs; jobs[k].size = size; jobs[k].qp = qp; jobs[k].coeff_type = coeff_type; jobs[k].fast = fast; }
      be.tx_multi(jobs, 2, bit);
      *bu = bit[0]; *bv = bit[1];
    } else {
      *bu = be.tx_chain(ou, os, pu, ps, ru, rs, cqu, size, qp, coeff_type, fast);
      *bv = be.tx_chain(ov, os, pv, ps, rv, rs, cqv, size, qp, coeff_type, fast);
    }
  }
  // encode_and_reconstruct_block_intra_uv :1170-1273; returns (cbp_u << 8) | cbp_v
  TBR_HD TBR_NI int enc_rec_intra_uv(const S *ou, const S *ov, int os, S *ru, S *rv, int rfs, int ypos, int xpos, int size, int qp, S *pu, S *pv, int16_t *cqu, int16_t *cqv,
                              S *rbu, S *rbv, int coeff_type, int tb_split, int intra_mode, int upright, int downleft, const S *pblock_y, const S *rec_y,
                              int rec_stride2) {
    const int fast = F.speed > 1;
    int cbp_u = 0, cbp_v = 0;
    if (tb_split) {
      const int s2 = size / 2;
      int index = 0;
      for (int i = 0; i < size; i += s2)
        for (int j = 0; j < size; j += s2) {
          be.intra_predict(pu + i * size + j, size, ru, rfs, rbu + i * size + j, size, i, j, ypos, xpos, s2, upright, downleft, 1, intra_mode);
          be.intra_predict(pv + i * size + j, size, rv, rfs, rbv + i * size + j, size, i, j, ypos, xpos, s2, upright, downleft, 1, intra_mode);
          if (pblock_y) be.cfl(pblock_y + i * size + j, pu + i * size + j, pv + i * size + j, rec_y + (i << 1) * rec_stride2 + (j << 1), s2 << 1, size << 1, rec_stride2);
          int bu, bv;
          uv_chains(ou + i * os + j, ov + i * os + j, os, pu + i * size + j, pv + i * size + j, size, rbu + i * size + j, rbv + i * size + j, size, cqu + index, cqv + index, s2, qp,
                    coeff_type, fast, &bu, &bv);
          cbp_u = (cbp_u << 1) + bu;
          cbp_v = (cbp_v << 1) + bv;
          index += 256;
        }
    } else {
      be.intra_predict(pu, size, ru, rfs, (const S *)nullptr, 0, 0, 0, ypos, xpos, size, upright, downleft, 0, intra_mode);
      be.intra_predict(pv, size, rv, rfs, (const S *)nullptr, 0, 0, 0, ypos, xpos, size, upright, downleft, 0, intra_mode);
      if (pblock_y) be.cfl(pblock_y, pu, pv, rec_y, size << 1, size << 1, rec_stride2);
      uv_chains(ou, ov, os, pu, pv, size, rbu, rbv, size, cqu, cqv, size, qp, coeff_type, fast, &cbp_u, &cbp_v);
    }
    return (cbp_u << 8) | cbp_v;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // encode_block :1340-1514 — evaluates candidate c into W.rec_* / W.cq_*, fills c.cbp_*, returns the bits write_block would emit.
  // (c.cbp_* keep the coded values; the deblocking values (1,1,1 when tb_split, :1494-1497) are applied by commit_block.)
  // ---------------------------------------------------------------------------------------------------------------
  TBR_HD TBR_NI int encode_block(const BlockInfo &bi, Cand &c) {
    const int size = bi.size, ypos = bi.ypos, xpos = bi.xpos, yc = ypos >> 1, xc = xpos >> 1, sizeC = size >> 1;
    const int tb_split = imax(0, c.tb_param), zero_block = c.tb_param == -1;
    c.tb_split = tb_split;
    const S *oy = F.org[0] + ypos * F.org_stride[0] + xpos, *ou = F.org[1] + yc * F.org_stride[1] + xc, *ov = F.org[2] + yc * F.org_stride[1] + xc;
    const int itype = (F.frame_type == I_FRAME) << 1;
    if (c.mode == MODE_INTRA) {
      const int ur = upright_available(ypos, xpos, size, size, F.width, F.height, F.sb_size), dl = downleft_available(ypos, xpos, size, size, F.width, F.height, F.sb_size);
      S *yrec = F.rec[0] + ypos * F.rec_stride[0] + xpos, *urec = F.rec[1] + yc * F.rec_stride[1] + xc, *vrec = F.rec[2] + yc * F.rec_stride[1] + xc;
      c.cbp_y = enc_rec_intra(oy, F.org_stride[0], yrec, F.rec_stride[0], ypos, xpos, size, F.qp, W.p_y, W.cq_y, W.rec_y, itype | 0, tb_split, c.intra_mode, ur, dl);
      const int uv = enc_rec_intra_uv(ou, ov, F.org_stride[1], urec, vrec, F.rec_stride[1], yc, xc, sizeC, F.qpc, W.p_u, W.p_v, W.cq_u, W.cq_v, W.rec_u, W.rec_v, itype | 1,
                                      tb_split && sizeC > 4, c.intra_mode, ur, dl, F.cfl_intra ? W.p_y : (const S *)nullptr, W.rec_y, size);
      c.cbp_u = uv >> 8; c.cbp_v = uv & 255;
    } else {
      if (!(reuse_pred && !F.cfl_inter)) predict_inter(bi, c);  // the reference predicts again for every tb_param of the same vectors: identical samples
      if (c.mode == MODE_SKIP || zero_block) {
        be.copy(W.rec_y, size, W.p_y, size, size, size);
        be.copy(W.rec_u, sizeC, W.p_u, sizeC, sizeC, sizeC);
        be.copy(W.rec_v, sizeC, W.p_v, sizeC, sizeC, sizeC);
        c.cbp_y = c.cbp_u = c.cbp_v = 0;
      } else {
        if (!F.cfl_inter && sizeC <= 8) {
          // small blocks: the chains of the three planes (<= 12 of 4x4 / 8x8, one thread each on the device) side by side; a 16x16 luma block goes first, alone
          TxJob<S> jobs[12];
          int bit[12], n = 0, ny = 0;
          const int tbc = tb_split && sizeC > 4;
          if (size == 16 && !tb_split) c.cbp_y = enc_rec_inter(oy, F.org_stride[0], size, F.qp, W.p_y, W.cq_y, W.rec_y, itype | 0, 0);
          else { ny = inter_jobs(jobs, oy, F.org_stride[0], size, F.qp, W.p_y, W.cq_y, W.rec_y, itype | 0, tb_split); n = ny; }
          const int nu = inter_jobs(jobs + n, ou, F.org_stride[1], sizeC, F.qpc, W.p_u, W.cq_u, W.rec_u, itype | 1, tbc);
          n += nu;
          const int nv = inter_jobs(jobs + n, ov, F.org_stride[1], sizeC, F.qpc, W.p_v, W.cq_v, W.rec_v, itype | 1, tbc);
          n += nv;
          be.tx_multi(jobs, n, bit);
          if (ny) c.cbp_y = join_cbp(bit, ny);
          c.cbp_u = join_cbp(bit + ny, nu);
          c.cbp_v = join_cbp(bit + ny + nu, nv);
        } else {
          c.cbp_y = enc_rec_inter(oy, F.org_stride[0], size, F.qp, W.p_y, W.cq_y, W.rec_y, itype | 0, tb_split);
          if (F.cfl_inter) be.cfl(W.p_y, W.p_u, W.p_v, W.rec_y, size, size, size);
          c.cbp_u = enc_rec_inter(ou, F.org_stride[1], sizeC, F.qpc, W.p_u, W.cq_u, W.rec_u, itype | 1, tb_split && sizeC > 4);
          c.cbp_v = enc_rec_inter(ov, F.org_stride[1], sizeC, F.qpc, W.p_v, W.cq_v, W.rec_v, itype | 1, tb_split && sizeC > 4);
        }
      }
    }
    return block_bits(bi, c, W.cq_y, W.cq_u, W.cq_v);
  }

  // cost_calc :916-926 (sub = 1)
  TBR_HD TBR_NI uint32_t cost_calc(const BlockInfo &bi, int width, int height, int nbits) {
    const int size = bi.size, yc = bi.ypos >> 1, xc = bi.xpos >> 1;
    const S *oy = F.org[0] + bi.ypos * F.org_stride[0] + bi.xpos, *ou = F.org[1] + yc * F.org_stride[1] + xc, *ov = F.org[2] + yc * F.org_stride[1] + xc;
    const uint64_t ssd = be.ssd(oy, F.org_stride[0], W.rec_y, size, width, height) + be.ssd(ou, F.org_stride[1], W.rec_u, size >> 1, width >> 1, height >> 1) +
                         be.ssd(ov, F.org_stride[1], W.rec_v, size >> 1, width >> 1, height >> 1);
    uint64_t cost = (ssd >> (F.bitdepth * 2 - 16)) + (uint64_t)(int64_t)mul_add_half(F.lambda, (double)nbits);
    if (cost > (1u << 30)) cost = 1u << 30;
    return (uint32_t)cost;
  }

  // copy_best_parameters :1615-1677
  TBR_HD TBR_NI void copy_best(BlockInfo &bi, const Cand &c) {
    const int size = bi.size, sc = size >> 1;
    be.copy(W.best_y, size, W.rec_y, size, size, size);
    be.copy(W.best_u, sc, W.rec_u, sc, sc, sc);
    be.copy(W.best_v, sc, W.rec_v, sc, sc, sc);
    if (c.cbp_y) be.copy_coeff(W.bq_y, W.cq_y);
    if (c.cbp_u) be.copy_coeff(W.bq_u, W.cq_u);
    if (c.cbp_v) be.copy_coeff(W.bq_v, W.cq_v);
    Cand &b = bi.best;
    b.pb_part = c.pb_part; b.skip_idx = c.skip_idx; b.mode = c.mode; b.cbp_y = c.cbp_y; b.cbp_u = c.cbp_u; b.cbp_v = c.cbp_v; b.tb_param = c.tb_param; b.tb_split = c.tb_split;
    if (c.mode == MODE_SKIP || c.mode == MODE_MERGE) {
      const IPred &p = c.mode == MODE_SKIP ? bi.skip_cand[c.skip_idx] : bi.merge_cand[c.skip_idx];
      b.ref_idx0 = p.ref_idx0; b.ref_idx1 = p.ref_idx1;
      for (int i = 0; i < 4; i++) { b.mv0[i] = p.mv0; b.mv1[i] = p.mv1; }
      b.dir = p.bipred_flag;
    } else if (c.mode == MODE_INTRA) {
      b.ref_idx0 = b.ref_idx1 = 0;
      for (int i = 0; i < 4; i++) { b.mv0[i].x = b.mv0[i].y = b.mv1[i].x = b.mv1[i].y = 0; }
      b.dir = -1; b.intra_mode = c.intra_mode;
    } else {
      b.ref_idx0 = c.ref_idx0; b.ref_idx1 = c.ref_idx1;
      for (int i = 0; i < 4; i++) { b.mv0[i] = c.mv0[i]; b.mv1[i] = c.mv1[i]; }
      b.dir = c.mode == MODE_INTER ? 0 : 2;
    }
  }

  // ---------------------------------------------------------------------------------------------------------------
  // searches
  // ---------------------------------------------------------------------------------------------------------------
  // search_inter_prediction_params :1033-1098.  org: block origin (pitch os), ref_idx selects the frame; candidates = W.mvcand[cand_ref]
  TBR_HD TBR_NI int search_inter(const S *org, int os, int ref_idx, const BlockInfo &bi, Mv mvc, Mv mvp, Mv *mv_arr, int part, int sign, int cand_ref) {
    const int size = bi.size, rs = F.ref_stride[0];
    const S *ref = F.ref[ref_idx][0] + bi.ypos * rs + bi.xpos;
    Mv mvp2 = mvp, mv;
    int sad = 0;
    const Mv *cand = W.mvcand[cand_ref];
    const int ncand = W.mvcand_num[cand_ref];
    if (part == PART_NONE) {
      sad += be.me(org, os, ref, rs, size, size, size, &mv, mvc, mvp2, F.sqrt_lambda, sign, bi.xpos, bi.ypos, cand, ncand);
      mv_arr[0] = mv_arr[1] = mv_arr[2] = mv_arr[3] = mv;
    } else if (part == PART_HOR) {
      for (int index = 0; index < 4; index += 2) {
        const int py = index >> 1;
        sad += be.me(org + py * (size / 2) * os, os, ref + py * (size / 2) * rs, rs, size, size, size / 2, &mv, mvc, mvp2, F.sqrt_lambda, sign, bi.xpos, bi.ypos, cand, ncand);
        mv_arr[index] = mv_arr[index + 1] = mv;
        mvp2 = mv_arr[0];
      }
    } else if (part == PART_VER) {
      for (int index = 0; index < 2; index++) {
        sad += be.me(org + index * (size / 2), os, ref + index * (size / 2), rs, size, size / 2, size, &mv, mvc, mvp2, F.sqrt_lambda, sign, bi.xpos, bi.ypos, cand, ncand);
        mv_arr[index] = mv_arr[index + 2] = mv;
        mvp2 = mv_arr[0];
      }
    } else {
      for (int index = 0; index < 4; index++) {
        const int px = index & 1, py = (index & 2) >> 1;
        sad += be.me(org + py * (size / 2) * os + px * (size / 2), os, ref + py * (size / 2) * rs + px * (size / 2), rs, size, size / 2, size / 2, &mv, mvc, mvp2,
                     F.sqrt_lambda, sign, bi.xpos, bi.ypos, cand, ncand);
        mv_arr[index] = mv;
        mvp2 = mv_arr[0];
      }
    }
    return sad;
  }

  // search_intra_prediction_params :928-1031 (SAD-based; order DC, HOR, VER, PLANAR, then the six angular modes)
  TBR_HD TBR_NI int search_intra(const BlockInfo &bi, int *intra_mode) {
    const int size = bi.size, ypos = bi.ypos, xpos = bi.xpos;
    const int ur = upright_available(ypos, xpos, size, size, F.width, F.height, F.sb_size), dl = downleft_available(ypos, xpos, size, size, F.width, F.height, F.sb_size);
    const S *oy = F.org[0] + ypos * F.org_stride[0] + xpos;
    S *yrec = F.rec[0] + ypos * F.rec_stride[0] + xpos;
    static const int8_t order[10] = {0 /*DC*/, 2 /*HOR*/, 3 /*VER*/, 1 /*PLANAR*/, 4, 5, 6, 7, 8, 9};
    int min_sad = 1 << 30;
    *intra_mode = 0;
    const int n = F.num_intra_modes == 4 ? 4 : 10;
    for (int k = 0; k < n; k++) {
      // search_intra_prediction_params calls get_dc_pred(left, top) directly (:951): unlike get_intra_prediction's DC it does not substitute the
      // other edge at xpos == 0 / ypos == 0 -> mode 10 = "DC from (left, top) as gathered"
      be.intra_predict(W.p_y, size, yrec, F.rec_stride[0], (const S *)nullptr, 0, 0, 0, ypos, xpos, size, ur, dl, 0, k == 0 ? 10 : order[k]);
      const int sad = (int)(be.sad(oy, F.org_stride[0], W.p_y, size, size, size) >> (F.bitdepth - 8));
      if (sad < min_sad) { *intra_mode = order[k]; min_sad = sad; }
    }
    return min_sad;
  }

  // search_bipred_prediction_params :1679-1833
  TBR_HD TBR_NI int search_bipred(const BlockInfo &bi, int part, const Mv *mv_center, Mv mvp, int *ref_idx0, int *ref_idx1, Mv *mv_arr0, Mv *mv_arr1, int me_mode) {
    const int size = bi.size;
    const S *oy = F.org[0] + bi.ypos * F.org_stride[0] + bi.xpos;
    if (me_mode) {
      const int r0 = F.interp_ref ? 1 : 0, r1 = F.interp_ref ? 2 : 1, rs = F.ref_stride[0];
      const S *ref0 = F.ref[r0][0] + bi.ypos * rs + bi.xpos, *ref1 = F.ref[r1][0] + bi.ypos * rs + bi.xpos;
      Mv mv;
      const int sad = be.me_bi(oy, F.org_stride[0], ref0, ref1, rs, size, &mv, mv_center[r0], mvp, F.sqrt_lambda, 0, bi.xpos, bi.ypos, W.mvcand[r0], W.mvcand_num[r0], W.p0_y, W.p1_y);
      // motion_estimate_bi scribbles on the caller's list (:873-881): entries num..3 are zeroed, [4] = mvp (quarter-pel, sic), [5] = 0; the
      // list length is unchanged, so entries 4 and 5 stay visible to every later search of this super block once the list is that long
      for (int idx = W.mvcand_num[r0]; idx < 4; idx++) { W.mvcand[r0][idx].x = 0; W.mvcand[r0][idx].y = 0; }
      W.mvcand[r0][4] = mvp; W.mvcand[r0][5].x = 0; W.mvcand[r0][5].y = 0;
      *ref_idx0 = r0; *ref_idx1 = r1;
      for (int i = 0; i < 4; i++) mv_arr0[i] = mv_arr1[i] = mv;
      return sad;
    }
    int min_ref_idx0 = (F.frame_type == B_FRAME && F.interp_ref > 0) ? 1 : 0, min_ref_idx1 = 0;
    Mv min0[4], min1[4], mv_all[4];
    for (int i = 0; i < 4; i++) min0[i] = min1[i] = mvp;
    int min_sad = 1 << 30;
    const int num_iter = F.speed == 0 ? 2 : 1;
    for (int n = 0; n < num_iter; n++) {
      const int stop = part == 0 ? 0 : 1;
      for (int list = 1; list >= stop; list--) {
        const Mv mv = list ? min0[0] : min1[0];
        int ref_idx = list ? min_ref_idx0 : min_ref_idx1;
        inter_pred_yuv(ref_idx, W.p_y, W.p_u, W.p_v, bi.ypos, bi.xpos, bi.size, bi.bwidth, bi.bheight, list ? min0 : min1, F.ref_sign[ref_idx], part > 0, 1);
        be.sat2ab(W.org8, oy, F.org_stride[0], W.p_y, size);
        int ref_start, ref_end;
        if (F.frame_type == P_FRAME) { ref_start = 0; ref_end = F.num_ref - 1; }
        else { ref_start = ref_end = (list ? 1 : 0) + (F.interp_ref ? 1 : 0); }
        for (ref_idx = ref_start; ref_idx <= ref_end; ref_idx++) {
          const Mv mvp2 = (F.frame_type == B_FRAME && list == 1) ? mv : mvp;
          const int sad = search_inter(W.org8, size, ref_idx, bi, mv_center[ref_idx], mvp2, mv_all, part, F.ref_sign[ref_idx], ref_idx);
          for (int i = 0; i < 4; i++) add_mvcandidate(mv_all[i], ref_idx);
          if (sad < min_sad) {
            min_sad = sad;
            if (list) { min_ref_idx1 = ref_idx; for (int i = 0; i < 4; i++) min1[i] = mv_all[i]; }
            else { min_ref_idx0 = ref_idx; for (int i = 0; i < 4; i++) min0[i] = mv_all[i]; }
          }
        }
      }
    }
    *ref_idx0 = min_ref_idx0; *ref_idx1 = min_ref_idx1;
    for (int i = 0; i < 4; i++) { mv_arr0[i] = min0[i]; mv_arr1[i] = min1[i]; }
    return min_sad / 2;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // mode_decision_rdo :1835-2120
  // ---------------------------------------------------------------------------------------------------------------
  TBR_HD void cand_group_begin() { cidx = 0; loc_idx = 0x7fffffff; loc_cost = MAX_U32; loc_worst = 0; loc_bestc = MAX_U32; }
  // candidate number cidx of the current group: evaluated by the warp that owns it; track_range: also the worst / best cost (:1998-1999)
  TBR_HD TBR_NI void try_cand(BlockInfo &bi, Cand &c, int w, int h, bool track_range = false) {
    const int my = cidx++;
    if (!be.mine(my)) return;
    const int nbits = encode_block(bi, c);
    const uint32_t cost = cost_calc(bi, w, h, nbits);
    if (track_range) { loc_worst = loc_worst > cost ? loc_worst : cost; loc_bestc = loc_bestc < cost ? loc_bestc : cost; }
    if (cost < loc_cost) { loc_cost = cost; loc_idx = my; copy_best(bi, c); }
  }
  // end of a group: the winner over all warps = min (cost, index); every warp receives its cost and parameters, `owner` holds its blocks
  TBR_HD uint32_t cand_group_end(BlockInfo &bi, int *owner) {
    uint32_t cost = loc_cost;
    int idx = loc_idx;
    *owner = be.reduce_best(&cost, &idx);
    be.bcast(&bi.best, (int)sizeof(Cand), *owner);
    return cost;
  }
  TBR_HD static void set_from_ipred(Cand &c, const IPred &p, int idx) {
    c.skip_idx = idx; c.ref_idx0 = p.ref_idx0; c.ref_idx1 = p.ref_idx1; c.mv0[0] = p.mv0; c.mv1[0] = p.mv1; c.dir = p.bipred_flag;
  }

  TBR_HD TBR_NI uint32_t mode_decision_serial(BlockInfo &bi, int *owner) {
    const int size = bi.size, ypos = bi.ypos, xpos = bi.xpos;
    const int rectangular = bi.bwidth != size || bi.bheight != size;
    const int intra_inter_sad = F.speed > 0;
    uint32_t sad_intra = MAX_U32;
    int do_inter = 1, do_intra = 1;
    cand_group_begin();
    Cand t;
    t.mode = MODE_SKIP; t.intra_mode = 0; t.skip_idx = 0; t.pb_part = PART_NONE; t.ref_idx0 = t.ref_idx1 = 0; t.dir = 0; t.cbp_y = t.cbp_u = t.cbp_v = 0; t.tb_param = 0; t.tb_split = 0;
    for (int i = 0; i < 4; i++) { t.mv0[i].x = t.mv0[i].y = t.mv1[i].x = t.mv1[i].y = 0; }
    int intra_mode = 0;

    if (F.frame_type != I_FRAME) {
      t.tb_param = 0; t.pb_part = PART_NONE; t.mode = MODE_SKIP;
      for (int k = 0; k < bi.num_skip; k++) {
        set_from_ipred(t, bi.skip_cand[k], k);
        t.mode = MODE_SKIP;
        try_cand(bi, t, bi.bwidth, bi.bheight);
      }
    }
    if ((size < 128 || F.speed == 0) && !rectangular && size <= MAX_TR) {
      if (F.frame_type != I_FRAME) {
        t.tb_param = 0;
        be.mark(PH_OTHER);
        for (int k = 0; k < bi.num_merge; k++) {
          set_from_ipred(t, bi.merge_cand[k], k);
          t.mode = MODE_MERGE;
          for (int tb = 0; tb <= bi.max_tb - 1; tb++) { t.tb_param = tb; try_cand(bi, t, size, size); }
        }
        if (intra_inter_sad) {
          sad_intra = (uint32_t)search_intra(bi, &intra_mode);
          sad_intra += (uint32_t)(int)mul_add_half(F.sqrt_lambda, 2.0);
        }
        t.mode = MODE_INTER;
        int min_idx, max_idx;
        if (best_ref < 0 || F.speed < 2 || F.enable_bipred) { min_idx = 0; max_idx = F.num_ref - 1; }
        else min_idx = max_idx = best_ref;
        if (F.frame_type == B_FRAME && F.interp_ref > 2) min_idx = 1;
        Mv mv_all[TB_RDO_MAX_REF][4][4], mv_center[TB_RDO_MAX_REF], mvp;
        uint32_t sad_inter_r[TB_RDO_MAX_REF];
        const S *oy = F.org[0] + ypos * F.org_stride[0] + xpos;
        be.mark(PH_SKIP_MERGE);
        mvp = get_mv_pred(ypos, xpos, size, size);  // the same for every reference (its ref_idx argument is unused, inter_prediction.c:413)
        bi.mvp = mvp;
        // (1) the searches: reference ref_idx on warp (ref_idx - min_idx) mod NW.  A reference's searches only read and extend ITS candidate list
        for (int ref_idx = min_idx; ref_idx <= max_idx; ref_idx++) {
          if (!be.mine(ref_idx - min_idx)) continue;
          add_mvcandidate(mvp, ref_idx);
          const int sign = F.ref_sign[ref_idx];
          mv_center[ref_idx] = mvp;
          uint32_t sad_inter = MAX_U32;
          for (int part = 0; part < bi.max_pb; part++) {
            const uint32_t sad = (uint32_t)search_inter(oy, F.org_stride[0], ref_idx, bi, mv_center[ref_idx], mvp, mv_all[ref_idx][part], part, sign, ref_idx);
            for (int i = 0; i < 4; i++) add_mvcandidate(mv_all[ref_idx][part][i], ref_idx);
            mv_center[ref_idx] = mv_all[ref_idx][0][0];
            sad_inter = sad_inter < sad ? sad_inter : sad;
          }
          sad_inter_r[ref_idx] = sad_inter;
          be.put_me(ref_idx, &mv_all[ref_idx][0][0], sad_inter);
        }
        be.cta_sync();
        // (2) every warp learns the other references' vectors and replays their effect on its replica of the candidate lists
        for (int ref_idx = min_idx; ref_idx <= max_idx; ref_idx++) {
          if (be.mine(ref_idx - min_idx)) continue;
          be.get_me(ref_idx, &mv_all[ref_idx][0][0], &sad_inter_r[ref_idx]);
          add_mvcandidate(mvp, ref_idx);
          for (int part = 0; part < bi.max_pb; part++)
            for (int i = 0; i < 4; i++) add_mvcandidate(mv_all[ref_idx][part][i], ref_idx);
          mv_center[ref_idx] = mv_all[ref_idx][0][0];
        }
        be.cta_sync();
        be.mark(PH_SEARCH);
        // (3) the RD candidates of every reference
        for (int ref_idx = min_idx; ref_idx <= max_idx; ref_idx++) {
          t.ref_idx0 = t.ref_idx1 = ref_idx;
          if (intra_inter_sad) {
            do_inter = sad_inter_r[ref_idx] < sad_intra;
            if (sad_inter_r[ref_idx] < sad_intra) do_intra = 0;
          }
          if (do_inter) {
            for (int part = 0; part < bi.max_pb; part++) {
              t.pb_part = part;
              for (int i = 0; i < 4; i++) t.mv0[i] = t.mv1[i] = mv_all[ref_idx][part][i];
              const int min_tb = F.speed < 1 ? -1 : 0;
              t.mode = MODE_INTER; t.dir = 0;
              for (int tb = min_tb; tb <= bi.max_tb - 1; tb++) {
                t.tb_param = tb;
                try_cand(bi, t, size, size, true);
              }
            }
          }
        }
        {
          uint32_t worst_cost = loc_worst, best_cost = loc_bestc;
          be.reduce_range(&worst_cost, &best_cost);
          if (worst_cost && (uint64_t)worst_cost * 3 > (uint64_t)best_cost * 4) best_ref = 0;  // best_ref_idx is never updated in the reference (:1868, :2019)
        }
        be.mark(PH_INTER_CAND);

        if (F.num_ref > 1 && F.enable_bipred && do_inter) {
          int r0, r1;
          Mv a0[4], a1[4];
          // BIPRED_PART = 0: one partition
          search_bipred(bi, 0, mv_center, mvp, &r0, &r1, a0, a1, 0);
          t.pb_part = 0; t.ref_idx0 = r0; t.ref_idx1 = r1;
          for (int i = 0; i < 4; i++) { t.mv0[i] = a0[i]; t.mv1[i] = a1[i]; }
          t.mode = MODE_BIPRED;
          for (int tb = 0; tb <= bi.max_tb - 1; tb++) { t.tb_param = tb; try_cand(bi, t, size, size); }
          if (F.frame_type == B_FRAME && F.speed == 0) {
            search_bipred(bi, 1, mv_center, mvp, &r0, &r1, a0, a1, 1);
            t.pb_part = PART_NONE; t.ref_idx0 = r0; t.ref_idx1 = r1;
            for (int i = 0; i < 4; i++) { t.mv0[i] = a0[i]; t.mv1[i] = a1[i]; }
            t.tb_param = 0; t.mode = MODE_BIPRED;
            try_cand(bi, t, size, size);
          }
        }
      }
      be.mark(PH_BIPRED);
      if (do_intra) {
        t.mode = MODE_INTRA;
        if (F.intra_rdo) {
          // choice of the intra mode by RD cost (:2080-2097): its own distributed group, no copy_best
          uint32_t min_intra_cost = MAX_U32;
          int best_k = 0x7fffffff, k = 0;
          for (int m = 0; m < F.num_intra_modes; m++) {
            t.intra_mode = m;
            for (int tb = 0; tb <= bi.max_tb - 1; tb++, k++) {
              if (!be.mine(k)) continue;
              t.tb_param = tb; t.mode = MODE_INTRA;
              const int nbits = encode_block(bi, t);
              const uint32_t cost = cost_calc(bi, size, size, nbits);
              if (cost < min_intra_cost) { min_intra_cost = cost; best_k = k; }
            }
          }
          be.reduce_best(&min_intra_cost, &best_k);
          intra_mode = min_intra_cost == MAX_U32 ? 0 : best_k / bi.max_tb;
        } else
          search_intra(bi, &intra_mode);
        t.intra_mode = intra_mode;
        be.mark(PH_INTRA_SEARCH);
        for (int tb = 0; tb <= bi.max_tb - 1; tb++) { t.tb_param = tb; t.mode = MODE_INTRA; try_cand(bi, t, size, size); }
      }
    }
    const uint32_t cost_ = cand_group_end(bi, owner);
    be.mark(PH_INTRA_CAND);
    return cost_;
  }


  // candidate `idx` (its position in the reference's evaluation order) evaluated by whichever warp calls this; the warp keeps its best (cost, idx)
  TBR_HD TBR_NI void eval_cand(BlockInfo &bi, Cand &c, int w, int h, int idx, bool track_range) {
    const int nbits = encode_block(bi, c);
    const uint32_t cost = cost_calc(bi, w, h, nbits);
    if (track_range) { loc_worst = loc_worst > cost ? loc_worst : cost; loc_bestc = loc_bestc < cost ? loc_bestc : cost; }
    if (cost < loc_cost || (cost == loc_cost && idx < loc_idx)) { loc_cost = cost; loc_idx = idx; copy_best(bi, c); }
  }
  // one item of the intra-mode search (:2080-2097 with intra_rdo, else search_intra_prediction_params): the warp keeps its best (cost, k)
  TBR_HD TBR_NI void intra_search_item(BlockInfo &bi, Cand &t, int k, uint32_t *best_cost, int *best_k) {
    if (F.intra_rdo) {
      t.intra_mode = k / bi.max_tb; t.tb_param = k % bi.max_tb; t.mode = MODE_INTRA;
      const int nbits = encode_block(bi, t);
      const uint32_t cost = cost_calc(bi, bi.size, bi.size, nbits);
      if (cost < *best_cost || (cost == *best_cost && k < *best_k)) { *best_cost = cost; *best_k = k; }
    } else {
      int mode;
      search_intra(bi, &mode);
      *best_cost = 0; *best_k = mode * bi.max_tb;
    }
  }

  // mode_decision_rdo for square blocks of inter frames at encoder_speed 0, with the sections of the decision that do not depend on each other
  // OVERLAPPED over the warps of the CTA instead of run one after the other:
  //   while the references' motion searches run (one warp per reference), the remaining warps start the intra-mode search;
  //   then ONE warp runs the bi-prediction chain (search_bipred_prediction_params: every search depends on the previous one) and evaluates its
  //   candidates, while the others draw the inter candidates and the rest of the intra-mode search from shared counters.
  // Every candidate keeps the index it has in the reference's evaluation order, so the winner = min (cost, index) is the reference's
  // "first candidate with the strictly smallest cost" whichever warp evaluated what.  The candidate lists the chain extends are copied to
  // the other warps' replicas afterwards.
  TBR_HD TBR_NI uint32_t mode_decision_overlap(BlockInfo &bi, int *owner) {
    const int size = bi.size, ypos = bi.ypos, xpos = bi.xpos, nw = be.nwarps();
    be.queue_reset();
    be.mark2(-1);
    cand_group_begin();
    Cand t;
    t.mode = MODE_SKIP; t.intra_mode = 0; t.skip_idx = 0; t.pb_part = PART_NONE; t.ref_idx0 = t.ref_idx1 = 0; t.dir = 0; t.cbp_y = t.cbp_u = t.cbp_v = 0; t.tb_param = 0; t.tb_split = 0;
    for (int i = 0; i < 4; i++) { t.mv0[i].x = t.mv0[i].y = t.mv1[i].x = t.mv1[i].y = 0; }
    be.mark(PH_OTHER);
    int idx = 0;
    for (int k = 0; k < bi.num_skip; k++, idx++) {
      if (!be.mine(idx)) continue;
      set_from_ipred(t, bi.skip_cand[k], k);
      t.mode = MODE_SKIP; t.tb_param = 0; t.pb_part = PART_NONE;
      eval_cand(bi, t, bi.bwidth, bi.bheight, idx, false);
    }
    for (int k = 0; k < bi.num_merge; k++) {  // the tb_param variants of one merge candidate share its prediction: same warp
      const bool my = be.mine(bi.num_skip + k);
      for (int tb = 0; tb <= bi.max_tb - 1; tb++, idx++) {
        if (!my) continue;
        set_from_ipred(t, bi.merge_cand[k], k);
        t.mode = MODE_MERGE; t.tb_param = tb; t.pb_part = PART_NONE;
        reuse_pred = tb > 0;
        eval_cand(bi, t, size, size, idx, false);
      }
      reuse_pred = false;
    }
    be.mark(PH_SKIP_MERGE);

    int min_idx = 0;
    const int max_idx = F.num_ref - 1;
    if (F.frame_type == B_FRAME && F.interp_ref > 2) min_idx = 1;
    const int nrs = max_idx - min_idx + 1;
    Mv mv_all[TB_RDO_MAX_REF][4][4], mv_center[TB_RDO_MAX_REF], mvp;
    uint32_t sad_inter_r[TB_RDO_MAX_REF];
    const S *oy = F.org[0] + ypos * F.org_stride[0] + xpos;
    mvp = get_mv_pred(ypos, xpos, size, size);
    bi.mvp = mvp;
    const int n_isearch = F.intra_rdo ? F.num_intra_modes * bi.max_tb : 1;
    uint32_t my_icost = MAX_U32;
    int my_ik = 0x7fffffff;
    // (1) the searches, one reference per warp; warps without a reference begin the intra-mode search
    for (int ref_idx = min_idx; ref_idx <= max_idx; ref_idx++) {
      if (!be.mine(ref_idx - min_idx)) continue;
      add_mvcandidate(mvp, ref_idx);
      const int sign = F.ref_sign[ref_idx];
      mv_center[ref_idx] = mvp;
      uint32_t sad_inter = MAX_U32;
      for (int part = 0; part < bi.max_pb; part++) {
        const uint32_t sad = (uint32_t)search_inter(oy, F.org_stride[0], ref_idx, bi, mv_center[ref_idx], mvp, mv_all[ref_idx][part], part, sign, ref_idx);
        for (int i = 0; i < 4; i++) add_mvcandidate(mv_all[ref_idx][part][i], ref_idx);
        mv_center[ref_idx] = mv_all[ref_idx][0][0];
        sad_inter = sad_inter < sad ? sad_inter : sad;
      }
      sad_inter_r[ref_idx] = sad_inter;
      be.put_me(ref_idx, &mv_all[ref_idx][0][0], sad_inter);
    }
    be.mark2(0);  // (diagnostics) own searches done
    if (be.warp() >= nrs)
      for (int k; (k = be.next(1)) < n_isearch;) intra_search_item(bi, t, k, &my_icost, &my_ik);
    be.mark2(1);  // intra items taken while the searches run
    be.cta_sync();
    be.mark2(2);  // wait for the slowest warp of the phase
    for (int ref_idx = min_idx; ref_idx <= max_idx; ref_idx++) {
      if (be.mine(ref_idx - min_idx)) continue;
      be.get_me(ref_idx, &mv_all[ref_idx][0][0], &sad_inter_r[ref_idx]);
      add_mvcandidate(mvp, ref_idx);
      for (int part = 0; part < bi.max_pb; part++)
        for (int i = 0; i < 4; i++) add_mvcandidate(mv_all[ref_idx][part][i], ref_idx);
      mv_center[ref_idx] = mv_all[ref_idx][0][0];
    }
    be.cta_sync();
    be.mark(PH_SEARCH);

    // (2) the bi-prediction chain on warp 0; inter candidates and the intra-mode search on everybody (warp 0 joins when its chain is done)
    const int ntb = bi.max_tb + 1;  // tb_param -1 (no residual), 0, .. max_tb - 1 (encoder_speed < 1, :1990)
    const int n_inter = nrs * bi.max_pb * ntb;
    const int IDX_INTER = 64, IDX_BIPRED = IDX_INTER + n_inter, IDX_INTRA = IDX_BIPRED + 8;
    const bool do_bipred = F.num_ref > 1 && F.enable_bipred;
    if (do_bipred && be.warp() == 0) {
      int r0, r1;
      Mv a0[4], a1[4];
      search_bipred(bi, 0, mv_center, mvp, &r0, &r1, a0, a1, 0);
      t.pb_part = 0; t.ref_idx0 = r0; t.ref_idx1 = r1; t.dir = 0;
      for (int i = 0; i < 4; i++) { t.mv0[i] = a0[i]; t.mv1[i] = a1[i]; }
      t.mode = MODE_BIPRED;
      for (int tb = 0; tb <= bi.max_tb - 1; tb++) { t.tb_param = tb; reuse_pred = tb > 0; eval_cand(bi, t, size, size, IDX_BIPRED + tb, false); }
      reuse_pred = false;
      if (F.frame_type == B_FRAME) {
        search_bipred(bi, 1, mv_center, mvp, &r0, &r1, a0, a1, 1);
        t.pb_part = PART_NONE; t.ref_idx0 = r0; t.ref_idx1 = r1;
        for (int i = 0; i < 4; i++) { t.mv0[i] = a0[i]; t.mv1[i] = a1[i]; }
        t.tb_param = 0; t.mode = MODE_BIPRED;
        eval_cand(bi, t, size, size, IDX_BIPRED + bi.max_tb, false);
      }
      be.mark(PH_BIPRED);
    }
    for (int g; (g = be.next(0)) < nrs * bi.max_pb;) {  // one draw = the tb_param variants of one (reference, partition): they share the prediction
      const int part = g % bi.max_pb, ref_idx = min_idx + g / bi.max_pb;
      t.ref_idx0 = t.ref_idx1 = ref_idx; t.pb_part = part;
      for (int i = 0; i < 4; i++) t.mv0[i] = t.mv1[i] = mv_all[ref_idx][part][i];
      t.mode = MODE_INTER; t.dir = 0;
      for (int v = 0; v < ntb; v++) {
        t.tb_param = v - 1;
        reuse_pred = v > 0;
        eval_cand(bi, t, size, size, IDX_INTER + g * ntb + v, true);
      }
      reuse_pred = false;
    }
    be.mark(PH_INTER_CAND);
    for (int k; (k = be.next(1)) < n_isearch;) intra_search_item(bi, t, k, &my_icost, &my_ik);
    be.mark(PH_INTRA_SEARCH);
    {
      uint32_t worst_cost = loc_worst, best_cost = loc_bestc;
      be.reduce_range(&worst_cost, &best_cost);
      if (worst_cost && (uint64_t)worst_cost * 3 > (uint64_t)best_cost * 4) best_ref = 0;
    }
    if (do_bipred) {  // warp 0's searches extended (and scribbled on, :873-881) the candidate lists: everybody's replica follows
      if (be.warp() != 0)
        for (int r = 0; r < F.num_ref; r++) {
          be.copy_words(W.mvcand[r], W0.mvcand[r], 64 * (int)sizeof(Mv) / 4);
          W.mvcand_num[r] = W0.mvcand_num[r]; W.mvcand_mask[r] = W0.mvcand_mask[r];
        }
      be.cta_sync();
    }
    be.reduce_best(&my_icost, &my_ik);
    const int intra_mode = my_icost == MAX_U32 ? 0 : my_ik / bi.max_tb;
    t.intra_mode = intra_mode;
    for (int tb = 0; tb <= bi.max_tb - 1; tb++) {
      if (!be.mine(tb)) continue;
      t.tb_param = tb; t.mode = MODE_INTRA;
      eval_cand(bi, t, size, size, IDX_INTRA + tb, false);
    }
    const uint32_t cost_ = cand_group_end(bi, owner);
    be.mark(PH_INTRA_CAND);
    return cost_;
  }

  TBR_HD uint32_t mode_decision_rdo(BlockInfo &bi, int *owner) {
    if (F.frame_type != I_FRAME && F.speed == 0 && bi.bwidth == bi.size && bi.bheight == bi.size && bi.size <= MAX_TR && be.nwarps() > 1)
      return mode_decision_overlap(bi, owner);
    return mode_decision_serial(bi, owner);
  }

  // ---------------------------------------------------------------------------------------------------------------
  // early skip :2123-2399
  // ---------------------------------------------------------------------------------------------------------------
  TBR_HD static int es_threshold(int qp, int tr_log2size, double rel) {  // check_early_skip_transform_coeff :2123-2145
    static const uint16_t gquant[6] = {26214, 23302, 20560, 18396, 16384, 14564};  // common/common_tables.c:74
    const int shift2 = 21 - tr_log2size + qp / 6;
    const double fql = (double)(1 << shift2) / (double)gquant[qp % 6];
    return (int)(rel * fql);
  }
  TBR_HD TBR_NI int check_early_skip_block(const BlockInfo &bi, const Cand &c) {
    const int size = bi.size, size0 = imin(size, EARLY_SKIP_BLOCK), size0c = size0 >> 1;
    float thr = F.early_skip_thr;
    if (F.speed > 1 && size == F.sb_size) thr += thr / 4;
    // luma: 2x2 average then (size0/2)-point transform, threshold 0.5*thr of the first quantiser level (:2147-2180); chroma: calc_cbp (:2214-2229)
    const int thr_y = es_threshold(F.qp, ilog2_(size0 / 2), 0.5 * thr);
    const int thr_c = es_threshold(F.qpc, 5, thr) << (F.bitdepth - 8);
    int significant = 0;
    for (int i = 0; i < size && !significant; i += size0)
      for (int j = 0; j < size && !significant; j += size0) {
        const int y = bi.ypos + i, x = bi.xpos + j, yc = y >> 1, xc = x >> 1;
        Mv m0[4], m1[4];
        m0[0] = c.mv0[0]; m1[0] = c.mv1[0];
        if (c.dir == 2) {
          inter_pred_yuv(c.ref_idx0, W.p0_y, W.p0_u, W.p0_v, y, x, size0, size0, size0, m0, F.ref_sign_ge[c.ref_idx0], 0);
          inter_pred_yuv(c.ref_idx1, W.p1_y, W.p1_u, W.p1_v, y, x, size0, size0, size0, m1, F.ref_sign_ge[c.ref_idx1], 0);
          be.avg(W.p_y, W.p0_y, W.p1_y, size0, size0, size0);
          be.avg(W.p_u, W.p0_u, W.p1_u, size0c, size0c, size0c);
          be.avg(W.p_v, W.p0_v, W.p1_v, size0c, size0c, size0c);
        } else
          inter_pred_yuv(c.ref_idx0, W.p_y, W.p_u, W.p_v, y, x, size0, size0, size0, m0, F.ref_sign[c.ref_idx0], 0);
        significant = be.es_luma(F.org[0] + y * F.org_stride[0] + x, F.org_stride[0], W.p_y, size0, size0, thr_y);
        if (!significant) significant = be.es_chroma(F.org[1] + yc * F.org_stride[1] + xc, F.org_stride[1], W.p_u, size0c, size0c, thr_c);
        if (!significant) significant = be.es_chroma(F.org[2] + yc * F.org_stride[1] + xc, F.org_stride[1], W.p_v, size0c, size0c, thr_c);
      }
    return !significant;
  }
  // :2352-2392.  Skip candidate k (its early-skip test and, if it passes, its RD cost) on warp k mod NW
  TBR_HD TBR_NI int search_early_skip(BlockInfo &bi, uint32_t *cost, int *owner) {
    int flag = 0;
    Cand t;
    t.intra_mode = 0; t.pb_part = PART_NONE; t.cbp_y = t.cbp_u = t.cbp_v = 0; t.tb_split = 0;
    for (int i = 0; i < 4; i++) { t.mv0[i].x = t.mv0[i].y = t.mv1[i].x = t.mv1[i].y = 0; }
    cand_group_begin();
    for (int k = 0; k < bi.num_skip; k++) {
      t.tb_param = 0;
      set_from_ipred(t, bi.skip_cand[k], k);
      t.mode = MODE_SKIP;
      if (be.mine(cidx)) {
        if (check_early_skip_block(bi, t)) { flag = 1; try_cand(bi, t, bi.size, bi.size); }
        else cidx++;
      } else cidx++;
    }
    flag = be.reduce_or(flag);
    // the reference encodes the chosen candidate once more (final_encode = 3) and returns that cost: same bits, same reconstruction, same cost
    *cost = cand_group_end(bi, owner);
    return flag;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // commit: copy_block_to_frame :1516 + copy_deblock_data :1568 + the leaf record (what the final write_block needs)
  // ---------------------------------------------------------------------------------------------------------------
  // Only warp `owner` (the one whose scratch holds the winning blocks) stores; every warp advances the leaf / coefficient counters; the CTA
  // barrier at the end publishes the block to the other warps (and, through the row's progress counter, to the other CTAs).
  TBR_HD TBR_NI void commit_block(const BlockInfo &bi, uint32_t cost, int owner, const S *by, const S *bu, const S *bv, const int16_t *qy, const int16_t *qu, const int16_t *qv) {
    const int size = bi.size, sc = size >> 1, bw = bi.bwidth, bh = bi.bheight;
    const Cand &b = bi.best;
    const bool has_coeff = b.mode != MODE_SKIP && (b.cbp_y || b.cbp_u || b.cbp_v);
    const int tbc_ = b.tb_split && sc > 4;
    const int ny_ = coeff_count(size, b.tb_split), nc_ = coeff_count(sc, tbc_);
    if (be.warp() != owner) {
      if (has_coeff) coeff_used += ny_ + 2 * nc_;
      n_leaves++;
      be.cta_sync();
      return;
    }
    be.copy(F.rec[0] + bi.ypos * F.rec_stride[0] + bi.xpos, F.rec_stride[0], by, size, bw, bh);
    be.copy(F.rec[1] + (bi.ypos >> 1) * F.rec_stride[1] + (bi.xpos >> 1), F.rec_stride[1], bu, sc, bw >> 1, bh >> 1);
    be.copy(F.rec[2] + (bi.ypos >> 1) * F.rec_stride[1] + (bi.xpos >> 1), F.rec_stride[1], bv, sc, bw >> 1, bh >> 1);
    const int tb_split = imax(0, b.tb_param);
    tb_rdo_blk_t v;
    v.mode = (uint8_t)b.mode; v.size = (uint8_t)size; v.tb_split = (uint8_t)tb_split; v.pb_part = (uint8_t)(b.mode == MODE_INTER ? b.pb_part : PART_NONE);
    // encode_block :1494-1497: with tb_split the stored cbp is (1,1,1) ("used for deblocking only")
    v.cbp_y = (uint8_t)(b.tb_split ? 1 : b.cbp_y); v.cbp_u = (uint8_t)(b.tb_split ? 1 : b.cbp_u); v.cbp_v = (uint8_t)(b.tb_split ? 1 : b.cbp_v);
    v.bipred_flag = (int8_t)b.dir; v.ref_idx0 = (uint8_t)b.ref_idx0; v.ref_idx1 = (uint8_t)b.ref_idx1; v.pad[0] = v.pad[1] = 0;
    be.store_blk(F.blk, F.blk_stride, bi.ypos / MIN_PB, bi.xpos / MIN_PB, bw / MIN_PB, bh / MIN_PB, size / (2 * MIN_PB), v, b.mv0, b.mv1);
    // leaf record
    tb_rdo_leaf_t L;
    L.xpos = (uint16_t)bi.xpos; L.ypos = (uint16_t)bi.ypos; L.size = (uint8_t)size; L.mode = (uint8_t)b.mode; L.intra_mode = (uint8_t)b.intra_mode; L.skip_idx = (uint8_t)b.skip_idx;
    L.pb_part = (uint8_t)b.pb_part; L.tb_split = (uint8_t)b.tb_split; L.ref_idx0 = (uint8_t)b.ref_idx0; L.ref_idx1 = (uint8_t)b.ref_idx1; L.dir = (int8_t)b.dir;
    L.cbp_y = (uint8_t)b.cbp_y; L.cbp_u = (uint8_t)b.cbp_u; L.cbp_v = (uint8_t)b.cbp_v;
    L.num_skip_vec = (uint8_t)bi.num_skip; L.num_merge_vec = (uint8_t)bi.num_merge; L.ctx_index = (int8_t)bi.ctx.index; L.ctx_cbp = (int8_t)bi.ctx.cbp;
    for (int i = 0; i < 4; i++) { L.mv_arr0[i] = b.mv0[i]; L.mv_arr1[i] = b.mv1[i]; }
    L.mvp = bi.mvp; L.cost = cost; L.coeff_ofs = -1;
    if (b.mode != MODE_SKIP && (b.cbp_y || b.cbp_u || b.cbp_v)) {
      const int tbc = b.tb_split && sc > 4;
      const int ny = coeff_count(size, b.tb_split), nc = coeff_count(sc, tbc);
      int16_t *dst = F.coeffs + (size_t)sb_index * TB_RDO_SB_COEFFS + coeff_used;
      L.coeff_ofs = coeff_used;
      be.pack_coeff(dst, qy, size, b.tb_split, b.cbp_y != 0);
      be.pack_coeff(dst + ny, qu, sc, tbc, b.cbp_u != 0);
      be.pack_coeff(dst + ny + nc, qv, sc, tbc, b.cbp_v != 0);
      coeff_used += ny + 2 * nc;
    }
    be.store_leaf(F.leaves + (size_t)sb_index * TB_RDO_MAX_LEAVES + n_leaves, L);
    n_leaves++;
    be.cta_sync();
  }

  // ---------------------------------------------------------------------------------------------------------------
  // process_block :2401-2565, iteratively (depth <= 5: 128 -> 8)
  // ---------------------------------------------------------------------------------------------------------------
  struct Frame_ {
    int size, ypos, xpos, stage, child, leaf_start, coeff_start, encode_this, encode_rect, top_down, owner;
    uint32_t cost, cost_small;
    BlockInfo bi;
  };

  TBR_HD uint32_t process_sb(int sbx, int sby) {
    static const uint16_t iq_8x8[52] = {6,   7,   8,   8,   10,  11,  12,  13,  15,  17,  19,  21,  24,  27,  30,  34,   38,   43,   48,   54,   60,   68,   76,   86,   96,   108,
                                        121, 136, 152, 171, 192, 216, 242, 272, 305, 342, 384, 431, 484, 543, 610, 684,  768,  862,  968,  1086, 1219, 1368, 1536, 1724, 1935, 2172};
    const int nsbx = (F.width + F.sb_size - 1) / F.sb_size;
    sb_index = sby * nsbx + sbx;
    n_leaves = 0; coeff_used = 0; best_ref = -1;
    for (int r = 0; r < F.num_ref; r++) { W.mvcand_num[r] = 0; W.mvcand_mask[r] = 0; }
    Frame_ st[6];
    int sp = 0;
    uint32_t ret = 0;
    bool have_ret = false;
    st[0].size = F.sb_size; st[0].ypos = sby * F.sb_size; st[0].xpos = sbx * F.sb_size; st[0].stage = 0;
    while (sp >= 0) {
      Frame_ &f = st[sp];
      const int size = f.size, ypos = f.ypos, xpos = f.xpos;
      if (f.stage == 0) {
        if (ypos + MIN_BLOCK > F.height || xpos + MIN_BLOCK > F.width) { ret = 0; have_ret = true; sp--; continue; }
        const int smaller = size > MIN_BLOCK;
        f.encode_this = ypos + size <= F.height && xpos + size <= F.width;
        f.encode_rect = !f.encode_this && F.frame_type != I_FRAME;
        f.top_down = size == 2 * MIN_BLOCK && f.encode_this && F.frame_type != I_FRAME && F.speed > 0;
        f.cost_small = 1u << 28; f.cost = 1u << 28; f.child = 0; f.owner = 0;
        f.leaf_start = n_leaves; f.coeff_start = coeff_used;
        BlockInfo &bi = f.bi;
        bi.size = size; bi.ypos = ypos; bi.xpos = xpos; bi.bwidth = imin(size, F.width - xpos); bi.bheight = imin(size, F.height - ypos);
        bi.max_tb = F.enable_tb_split == 1 ? 2 : 1; bi.max_pb = F.enable_pb_split ? 4 : 1;
        bi.mvp.x = bi.mvp.y = 0;
        bi.num_skip = bi.num_merge = 0;
        bi.ctx = find_block_contexts(ypos, xpos, size);
        if (F.frame_type != I_FRAME && (f.encode_this || f.encode_rect)) {
          bi.num_skip = get_mv_skip_merge(ypos, xpos, size, size, bi.skip_cand);
          bi.num_merge = get_mv_skip_merge(ypos, xpos, size, size, bi.merge_cand);
        }
        if (f.encode_this && F.frame_type != I_FRAME && F.early_skip_thr > 0.0f) {
          uint32_t cost;
          int owner;
          be.mark(PH_OTHER);
          const int es = search_early_skip(bi, &cost, &owner);
          be.mark(PH_EARLY_SKIP);
          if (es) {
            commit_block(bi, cost, owner, W.best_y, W.best_u, W.best_v, W.bq_y, W.bq_u, W.bq_v);
            be.mark(PH_COMMIT);
            ret = cost; have_ret = true; sp--; continue;
          }
        }
        if (smaller && !f.top_down) { f.cost_small = 0; f.stage = 1; f.child = 0; }
        else f.stage = 2;
        continue;
      }
      if (f.stage == 1 || f.stage == 3) {  // children: TL, BL, TR, BR (:2513-2516)
        if (have_ret) { f.cost_small += ret; have_ret = false; f.child++; }
        if (f.child < 4) {
          const int ns = size / 2, k = f.child;
          Frame_ &c = st[sp + 1];
          c.size = ns; c.ypos = ypos + ((k & 1) ? ns : 0); c.xpos = xpos + ((k & 2) ? ns : 0); c.stage = 0;
          sp++;
        } else f.stage = f.stage == 1 ? 2 : 4;
        continue;
      }
      if (f.stage == 2) {
        if (f.encode_this || f.encode_rect) {
          f.cost = mode_decision_rdo(f.bi, &f.owner);
          const uint32_t thr = (uint32_t)(size * size * iq_8x8[F.qp] / 8);
          if (f.top_down && f.cost > thr) {
            // the children reuse the scratch blocks: the owner keeps this block's best aside in the CTA-shared save area (16x16 only)
            if (be.warp() == f.owner) {
              const int sc = size >> 1;
              be.copy(W0.td_y, size, W.best_y, size, size, size); be.copy(W0.td_u, sc, W.best_u, sc, sc, sc); be.copy(W0.td_v, sc, W.best_v, sc, sc, sc);
              be.copy_coeff(W0.tdq_y, W.bq_y); be.copy_coeff(W0.tdq_u, W.bq_u); be.copy_coeff(W0.tdq_v, W.bq_v);
            }
            be.cta_sync();
            f.cost_small = 0; f.stage = 3; f.child = 0;
            continue;
          }
        }
        f.stage = 4;
        continue;
      }
      // stage 4: choose between this size and the split (:2527-2546)
      if ((f.encode_this || f.encode_rect) && f.cost <= f.cost_small) {
        n_leaves = f.leaf_start; coeff_used = f.coeff_start;  // the children's blocks are replaced
        const bool from_td = f.top_down && f.child == 4;      // the children ran after this block's decision
        be.mark(PH_OTHER);
        if (from_td) commit_block(f.bi, f.cost, 0, W0.td_y, W0.td_u, W0.td_v, W0.tdq_y, W0.tdq_u, W0.tdq_v);
        else commit_block(f.bi, f.cost, f.owner, W.best_y, W.best_u, W.best_v, W.bq_y, W.bq_u, W.bq_v);
        be.mark(PH_COMMIT);
      }
      ret = f.cost < f.cost_small ? f.cost : f.cost_small; have_ret = true; sp--;
    }
    if (be.warp() == 0) be.store_count(F.leaf_count + sb_index, n_leaves);
    be.cta_sync();
    return ret;
  }
};

}  // namespace tbr
