// tb_api.cu — host side of libthor_b200.so: context, HBM-resident frames, batched entry points (tb_*), and the
// drop-in reference symbols (SURVEY.md §8b) that stage caller-owned host buffers through HBM per call.
// No CPU fallback anywhere: if CUDA is unusable the tb_* calls return TB_ERR_CUDA and the drop-in symbols abort
// (they have no error channel; the reference's own failure mode is fatalerror() -> abort(), common/global.h:38-44).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "tb_kernels.cuh"
#include "tb_tinterp.cuh"
#include <cmath>

using namespace tb;

// ---------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------
namespace {
struct Ctx {
  bool ready = false, failed = false;
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  uint64_t launches = 0;
  char err[512] = {0};
  static constexpr int NSLOT = 8;  // 0-3 operand windows, 4-6 compact copies, 7 filter flags
  void *slot[NSLOT] = {nullptr};
  size_t cap[NSLOT] = {0};
  int sm_count = 148;
  unsigned long long *me_stats = nullptr;
};
Ctx g;

void set_err(const char *what, cudaError_t e) { snprintf(g.err, sizeof(g.err), "%s: %s", what, cudaGetErrorString(e)); }

bool ensure_ctx() {
  if (g.ready) return true;
  if (g.failed) return false;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_err("thor_b200: no CUDA device", e == cudaSuccess ? cudaErrorNoDevice : e);
    g.failed = true;
    return false;
  }
  int dev = g.device;
  if (dev < 0 || dev >= n) dev = 0;
  if ((e = cudaSetDevice(dev)) != cudaSuccess) { set_err("cudaSetDevice", e); g.failed = true; return false; }
  g.device = dev;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) g.sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking)) != cudaSuccess) { set_err("cudaStreamCreate", e); g.failed = true; return false; }
  g.own_stream = true;
  {  // stream-ordered scratch (cudaMallocAsync) stays cached in the pool across synchronisations instead of going back to the driver
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      uint64_t keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  g.ready = true;
  return true;
}
[[noreturn]] void die(const char *where) {
  fprintf(stderr, "Run-time error...\nthor_b200 (%s): %s\n...now exiting to system...\n", where, g.err[0] ? g.err : "CUDA unavailable");
  abort();
}
inline void need_ctx(const char *where) {
  if (!ensure_ctx()) die(where);
}
inline void ck(cudaError_t e, const char *where) {
  if (e != cudaSuccess) { set_err(where, e); die(where); }
}
// the batched (B) entry points promise TB_ERR_CUDA, not abort(): only the drop-in symbols (no error channel in the reference's ABI) die
#define CKB(x, where)                                                        \
  do {                                                                       \
    cudaError_t e__ = (x);                                                   \
    if (e__ != cudaSuccess) { set_err(where, e__); return TB_ERR_CUDA; }     \
  } while (0)
void *slot_buf(int s, size_t bytes) {
  if (g.cap[s] < bytes) {
    if (g.slot[s]) { ck(cudaStreamSynchronize(g.stream), "sync"); cudaFree(g.slot[s]); }
    size_t c = bytes < (1u << 16) ? (1u << 16) : bytes * 2;
    ck(cudaMalloc(&g.slot[s], c), "cudaMalloc(stage)");
    g.cap[s] = c;
  }
  return g.slot[s];
}
inline int grid_for_warps(int nwarps) {  // persistent-style grid: a multiple of the SM count, capped by the work
  int ctas = (nwarps + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
  int cap = g.sm_count * 16;  // 16 CTAs x 4 warps = 64 resident warps per SM
  return ctas < 1 ? 1 : (ctas > cap ? cap : ctas);
}
#define LAUNCH(kernel, grid, block, smem, ...)                      \
  do {                                                              \
    kernel<<<(grid), (block), (smem), g.stream>>>(__VA_ARGS__);     \
    g.launches++;                                                   \
  } while (0)

// A 2-D window of a caller-owned host array staged in HBM so that device code can use the caller's indexing:
// dev()[y * dstride + x] <-> host[y * stride + x] for x0 <= x < x1, y0 <= y < y1 (element units).
struct Win {
  char *base = nullptr;
  const char *host = nullptr;
  int esz = 1, stride = 0, x0 = 0, y0 = 0, x1 = 0, y1 = 0;
  size_t pitch = 0;
  int dstride() const { return (int)(pitch / esz); }
  void *dev() const { return base - (ptrdiff_t)y0 * (ptrdiff_t)pitch - (ptrdiff_t)x0 * esz; }
};
Win win(int s, const void *host, int esz, int stride, int x0, int y0, int x1, int y1, bool upload) {
  Win w;
  // the window starts at device offset 0 of a 256-byte aligned slot: operands whose window starts at x0 = 0 (original
  // blocks, transform buffers) keep their alignment; halo windows (x0 < 0) are only read with alignment-agnostic loads
  const int x0r = x0;
  w.esz = esz; w.stride = stride; w.x0 = x0r; w.y0 = y0; w.x1 = x1; w.y1 = y1; w.host = (const char *)host;
  w.pitch = (((size_t)(x1 - x0r) * esz + 4) + 15) & ~(size_t)15;  // +4: ldw_any may touch the next word
  w.base = (char *)slot_buf(s, w.pitch * (size_t)(y1 - y0) + 64);
  if (upload)
    ck(cudaMemcpy2DAsync(w.base, w.pitch, w.host + ((ptrdiff_t)y0 * stride + x0r) * esz, (size_t)stride * esz, (size_t)(x1 - x0r) * esz, (size_t)(y1 - y0),
                         cudaMemcpyHostToDevice, g.stream), "H2D");
  return w;
}
void win_download(const Win &w, void *host_dst, int cx0, int cy0, int cx1, int cy1) {  // copy [cx0,cx1) x [cy0,cy1) back
  ck(cudaMemcpy2DAsync((char *)host_dst + ((ptrdiff_t)cy0 * w.stride + cx0) * w.esz, (size_t)w.stride * w.esz,
                       (char *)w.dev() + (ptrdiff_t)cy0 * (ptrdiff_t)w.pitch + (ptrdiff_t)cx0 * w.esz, w.pitch, (size_t)(cx1 - cx0) * w.esz, (size_t)(cy1 - cy0),
                       cudaMemcpyDeviceToHost, g.stream), "D2H");
}
inline void sync() { ck(cudaStreamSynchronize(g.stream), "cudaStreamSynchronize"); }
template <class T> T fetch(const void *dev) {
  T v;
  ck(cudaMemcpyAsync(&v, dev, sizeof(T), cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
  return v;
}

int chroma_qp_of(int qp) {  // common/common_tables.c:65-70
  static const int8_t mid[13] = {29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37};
  return qp < 30 ? qp : (qp >= 43 ? qp - 6 : mid[qp - 30]);
}
const uint8_t h_beta[52] = {0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15,
                            16, 17, 18, 20, 22, 24, 26, 28, 30, 32, 34, 36, 38, 40, 42, 44, 46, 48, 50, 52, 54, 56, 58, 60, 62, 64};
const uint8_t h_tc[56] = {0,  0,  1,  1,  2,  3,  4,  5,  6,  7,  8,  9,  10,  11,  12,  13,  14,  15,  16,
                          17, 18, 20, 22, 24, 26, 28, 30, 32, 36, 40, 44, 48,  52,  56,  60,  64,  68,  72,
                          80, 88, 96, 104, 112, 128, 144, 152, 160, 168, 176, 184, 192, 200, 208, 216, 224, 232};
}  // namespace

struct tb_frame {
  int width, height, pad, esz;
  int stride[3], pw[3], ph[3], padh[3], padv[3];
  void *base[3];
  void *origin[3];
  size_t bytes[3];
};
// layout of the reference's yuv_frame_t (common/types.h:58-80)
struct tb_yuv_frame {
  void *y, *u, *v;
  int width, height, stride_y, stride_c, offset_y, offset_c, pad_hor_y, pad_hor_c, pad_ver_y, pad_ver_c, area_y, area_c, sub, subsample, frame_num, bitdepth,
      input_bitdepth;
};

#define API_BEGIN() \
  if (!ensure_ctx()) return TB_ERR_CUDA;
#define API_END()                                              \
  do {                                                         \
    cudaError_t e__ = cudaGetLastError();                      \
    if (e__ != cudaSuccess) { set_err("kernel launch", e__); return TB_ERR_CUDA; } \
    return TB_OK;                                              \
  } while (0)

// ---- templated launch helpers of the frame-level entry points
template <class S> static void deblock_t(tb_frame *f, const tb_blkinfo_t *bi, int qp, int bitdepth) {
  const int w = f->width, h = f->height, maxv = (1 << bitdepth) - 1;
  // beta and tc are SAMPLE-typed in the reference (common/common_frame.c:68-69): truncate accordingly
  const int beta = (S)(h_beta[qp] << (bitdepth - 8));
  const int tc = (S)(bitdepth > 12 ? h_tc[qp] << (bitdepth - 12) : h_tc[qp] >> (12 - bitdepth));
  const int qpc = chroma_qp_of(qp);
  const int tcc = (S)(bitdepth > 12 ? h_tc[qpc] << (bitdepth - 12) : h_tc[qpc] >> (12 - bitdepth));
  S *Y = (S *)f->origin[0], *U = (S *)f->origin[1], *V = (S *)f->origin[2];
  {
    dim3 blk(32, 4), grd((w / 8 - 1 + 31) / 32 > 0 ? (w / 8 - 1 + 31) / 32 : 1, (h / 8 + 3) / 4);
    LAUNCH(deblock_y_vert_kernel<S>, grd, blk, 0, Y, f->stride[0], bi, w, h, beta, tc, maxv);
  }
  if (h > 8) {
    dim3 blk(128), grd((w + 127) / 128, h / 8 - 1 + ((h & 7) ? 1 : 0));
    LAUNCH(deblock_y_horz_kernel<S>, grd, blk, 0, Y, f->stride[0], bi, w, h, beta, tc, maxv);
  }
  {
    dim3 blk(32, 4), grd((w / 8 - 1 + 31) / 32 > 0 ? (w / 8 - 1 + 31) / 32 : 1, ((h >> 1) + 3) / 4, 2);
    LAUNCH(deblock_uv_kernel<S>, grd, blk, 0, U, V, f->stride[1], bi, w, h, 0, tcc, maxv);
  }
  if (h > 8) {
    dim3 blk(128), grd(((w >> 1) + 127) / 128, h / 8 - 1 + ((h & 7) ? 1 : 0), 2);
    LAUNCH(deblock_uv_kernel<S>, grd, blk, 0, U, V, f->stride[1], bi, w, h, 1, tcc, maxv);
  }
}
static void swap_plane(tb_frame *a, tb_frame *b, int p) {
  void *t = a->base[p]; a->base[p] = b->base[p]; b->base[p] = t;
  t = a->origin[p]; a->origin[p] = b->origin[p]; b->origin[p] = t;
}
static bool same_geometry(const tb_frame *a, const tb_frame *b) {
  return a->width == b->width && a->height == b->height && a->pad == b->pad && a->esz == b->esz;
}

template <class S>
static void clpf_t(tb_frame *rec, tb_frame *scr, const tb_blkinfo_t *bi, const uint8_t *fb_on, int fbl, int strength, int bitdepth, int plane, int qp) {
  const int sub = plane ? 1 : 0, pw = rec->pw[plane], ph = rec->ph[plane];
  const int nfb = ((pw + (1 << fbl) - 1) >> fbl) * ((ph + (1 << fbl) - 1) >> fbl);
  uint8_t *allskip = (uint8_t *)slot_buf(7, (size_t)nfb);
  LAUNCH(clpf_allskip_kernel, (nfb + 127) / 128, 128, 0, bi, pw, ph, sub, fbl, allskip);
  const int damping = bitdepth - 4 - (plane != 0) + (qp >> 4);
  dim3 blk(32, 8), grd((pw + 31) / 32, (ph + 7) / 8);
  LAUNCH(clpf_plane_kernel<S>, grd, blk, 0, (const S *)rec->origin[plane], (S *)scr->origin[plane], rec->stride[plane], pw, ph, bi, sub, allskip,
         plane == 0 ? fb_on : nullptr, fbl, strength << (bitdepth - 8), damping);
  swap_plane(rec, scr, plane);
}
template <class S>
static void cdef_t(tb_frame *rec, tb_frame *scr, const tb_blkinfo_t *bi, const int8_t *pri, const int8_t *sec, int pd, int sd, int32_t *dirvar, int bitdepth,
                   int plane) {
  const int w = rec->width, h = rec->height, nfb = ((w + 63) >> 6) * ((h + 63) >> 6), cs = bitdepth - 8;
  uint8_t *allskip = (uint8_t *)slot_buf(7, (size_t)nfb);
  LAUNCH(cdef_allskip_kernel, (nfb + 127) / 128, 128, 0, bi, w, h, allskip);
  if (plane == 0) {
    int nb = ((w + 7) >> 3) * ((h + 7) >> 3);
    LAUNCH(cdef_dir_kernel<S>, grid_for_warps(nb), CTA_THREADS, 0, (const S *)rec->origin[0], rec->stride[0], w, h, allskip, cs, dirvar);
  }
  const int sub = plane ? 1 : 0, pw = rec->pw[plane], ph = rec->ph[plane];
  dim3 blk(32, 8), grd((pw + 31) / 32, (ph + 7) / 8);
  LAUNCH(cdef_plane_kernel<S>, grd, blk, 0, (const S *)rec->origin[plane], (S *)scr->origin[plane], rec->stride[plane], w, h, pw, ph, sub, plane, bi, allskip, pri,
         sec, pd, sd, dirvar, cs);
  swap_plane(rec, scr, plane);
}
template <class S>
static void cdef_search_t(const tb_frame *rec, const tb_frame *org, const tb_blkinfo_t *bi, int speed, int pri_damping, int bitdepth, int32_t *dirvar, uint8_t *allskip,
                          uint64_t *mse) {
  static const int pristrengths[3] = {64, 32, 16};
  const int w = rec->width, h = rec->height, nfb = ((w + 63) >> 6) * ((h + 63) >> 6), cs = bitdepth - 8, total = pristrengths[speed];
  LAUNCH(cdef_allskip_kernel, (nfb + 127) / 128, 128, 0, bi, w, h, allskip);
  const int nb = ((w + 7) >> 3) * ((h + 7) >> 3);
  LAUNCH(cdef_dir_kernel<S>, grid_for_warps(nb), CTA_THREADS, 0, (const S *)rec->origin[0], rec->stride[0], w, h, allskip, cs, dirvar);
  ck(cudaMemsetAsync(mse, 0, sizeof(uint64_t) * 2 * (size_t)nfb * 64, g.stream), "memset");
  LAUNCH(cdef_search_kernel<S>, grid_for_warps(nfb * 2 * total), CTA_THREADS, 0, (const S *)rec->origin[0], (const S *)rec->origin[1], (const S *)rec->origin[2],
         (const S *)org->origin[0], (const S *)org->origin[1], (const S *)org->origin[2], rec->stride[0], rec->stride[1], w, h, bi, allskip, dirvar, speed, total,
         pri_damping, cs, (unsigned long long *)mse);
}
template <class S> static void pad_t(tb_frame *dst, const tb_frame *src, int border_only) {
  for (int p = 0; p < 3; p++) {
    dim3 blk(32, 8), grd((dst->pw[p] + 2 * dst->padh[p] + 31) / 32, (dst->ph[p] + 2 * dst->padv[p] + 7) / 8);
    LAUNCH(pad_copy_kernel<S>, grd, blk, 0, (S *)dst->origin[p], dst->stride[p], (const S *)src->origin[p], src->stride[p], dst->pw[p], dst->ph[p], dst->padh[p],
           dst->padv[p], border_only);
  }
}

extern "C" {

// ---------------------------------------------------------------------------------------------------------------
// management
// ---------------------------------------------------------------------------------------------------------------
int tb_init(int device) {
  if (!g.ready && !g.failed) {
    if (device < 0) {
      const char *lr = getenv("LOCAL_RANK");
      device = lr ? atoi(lr) : 0;
    }
    g.device = device;
  }
  return ensure_ctx() ? TB_OK : TB_ERR_CUDA;
}
const char *tb_last_error(void) { return g.err; }
uint64_t tb_launch_count(void) { return g.launches; }
void *tb_stream(void) { return ensure_ctx() ? (void *)g.stream : nullptr; }
int tb_set_stream(void *s) {
  API_BEGIN();
  if (g.own_stream) { cudaStreamSynchronize(g.stream); cudaStreamDestroy(g.stream); g.own_stream = false; }
  g.stream = (cudaStream_t)s;
  return TB_OK;
}
int tb_sync(void) {
  API_BEGIN();
  cudaError_t e = cudaStreamSynchronize(g.stream);
  if (e != cudaSuccess) { set_err("sync", e); return TB_ERR_CUDA; }
  return TB_OK;
}
void *tb_malloc(size_t bytes) {
  if (!ensure_ctx()) return nullptr;
  void *p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}
void tb_free(void *p) { if (p) cudaFree(p); }
int tb_memcpy_h2d(void *d, const void *s, size_t n) {
  API_BEGIN();
  cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, g.stream);
  if (e != cudaSuccess) { set_err("H2D", e); return TB_ERR_CUDA; }
  return TB_OK;
}
int tb_memcpy_d2h(void *d, const void *s, size_t n) {
  API_BEGIN();
  cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, g.stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
  if (e != cudaSuccess) { set_err("D2H", e); return TB_ERR_CUDA; }
  return TB_OK;
}
int tb_memcpy_d2h_async(void *d, const void *s, size_t n) {
  API_BEGIN();
  cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, g.stream);
  if (e != cudaSuccess) { set_err("D2H", e); return TB_ERR_CUDA; }
  return TB_OK;
}
int tb_memcpy_d2d(void *d, const void *s, size_t n) {
  API_BEGIN();
  cudaError_t e = cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, g.stream);
  if (e != cudaSuccess) { set_err("D2D", e); return TB_ERR_CUDA; }
  return TB_OK;
}
void *tb_malloc_host(size_t bytes) {
  if (!ensure_ctx()) return nullptr;
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}
void tb_free_host(void *p) { if (p) cudaFreeHost(p); }

// ---------------------------------------------------------------------------------------------------------------
// frames
// ---------------------------------------------------------------------------------------------------------------
tb_frame_t *tb_frame_create(int width, int height, int pad, int sample_bytes) {
  if (!ensure_ctx() || (sample_bytes != 1 && sample_bytes != 2) || width <= 0 || height <= 0) return nullptr;
  tb_frame *f = new tb_frame();
  f->width = width; f->height = height; f->pad = pad; f->esz = sample_bytes;
  for (int p = 0; p < 3; p++) {
    int sub = p ? 1 : 0;
    f->pw[p] = width >> sub; f->ph[p] = height >> sub; f->padh[p] = pad >> sub; f->padv[p] = pad >> sub;
    f->stride[p] = (f->pw[p] + 2 * f->padh[p] + 15) & ~15;
    f->bytes[p] = ((size_t)(f->ph[p] + 2 * f->padv[p]) * f->stride[p] + 64) * sample_bytes;
    if (cudaMalloc(&f->base[p], f->bytes[p]) != cudaSuccess) {
      for (int q = 0; q < p; q++) cudaFree(f->base[q]);  // the planes already allocated
      delete f;
      return nullptr;
    }
    cudaMemsetAsync(f->base[p], 0, f->bytes[p], g.stream);
    f->origin[p] = (char *)f->base[p] + ((size_t)f->padv[p] * f->stride[p] + f->padh[p]) * sample_bytes;
  }
  return f;
}
void tb_frame_destroy(tb_frame_t *f) {
  if (!f) return;
  for (int p = 0; p < 3; p++) cudaFree(f->base[p]);
  delete f;
}
int tb_frame_upload(tb_frame_t *f, const void *y, int ys, const void *u, const void *v, int cs) {
  API_BEGIN();
  const void *src[3] = {y, u, v};
  for (int p = 0; p < 3; p++) {
    if (!src[p]) continue;
    cudaError_t e = cudaMemcpy2DAsync(f->origin[p], (size_t)f->stride[p] * f->esz, src[p], (size_t)(p ? cs : ys) * f->esz, (size_t)f->pw[p] * f->esz, f->ph[p],
                                      cudaMemcpyDefault, g.stream);  // the source may be host (pinned or pageable) or device memory (UVA)
    if (e != cudaSuccess) { set_err("frame upload", e); return TB_ERR_CUDA; }
  }
  return TB_OK;
}
static int frame_download(const tb_frame *f, void *y, int ys, void *u, void *v, int cs, bool sync);
int tb_frame_download(const tb_frame_t *f, void *y, int ys, void *u, void *v, int cs) { return frame_download(f, y, ys, u, v, cs, true); }
int tb_frame_download_async(const tb_frame_t *f, void *y, int ys, void *u, void *v, int cs) { return frame_download(f, y, ys, u, v, cs, false); }
static int frame_download(const tb_frame *f, void *y, int ys, void *u, void *v, int cs, bool sync) {
  API_BEGIN();
  void *dst[3] = {y, u, v};
  for (int p = 0; p < 3; p++) {
    if (!dst[p]) continue;
    cudaError_t e = cudaMemcpy2DAsync(dst[p], (size_t)(p ? cs : ys) * f->esz, f->origin[p], (size_t)f->stride[p] * f->esz, (size_t)f->pw[p] * f->esz, f->ph[p],
                                      cudaMemcpyDefault, g.stream);
    if (e != cudaSuccess) { set_err("frame download", e); return TB_ERR_CUDA; }
  }
  cudaError_t e = sync ? cudaStreamSynchronize(g.stream) : cudaSuccess;
  if (e != cudaSuccess) { set_err("frame download", e); return TB_ERR_CUDA; }
  return TB_OK;
}
void *tb_frame_plane(const tb_frame_t *f, int plane, int *stride) {
  if (!f || plane < 0 || plane > 2) return nullptr;
  if (stride) *stride = f->stride[plane];
  return f->origin[plane];
}

// ---------------------------------------------------------------------------------------------------------------
// batched block-level entry points
// ---------------------------------------------------------------------------------------------------------------
int tb_sad_batch(const tb_sad_item_t *items, int n, int sample_bytes, int kind, uint32_t *out, int32_t *out2, uint64_t *out64) {
  API_BEGIN();
  if (sample_bytes != 1 && sample_bytes != 2) { set_err("tb_sad_batch: sample_bytes must be 1 or 2", cudaSuccess); return TB_ERR_ARG; }
  if (n <= 0) return TB_OK;
  if (sample_bytes == 1) LAUNCH(sad_batch_kernel<uint8_t>, grid_for_warps(n), CTA_THREADS, 0, items, n, kind, out, out2, out64);
  else LAUNCH(sad_batch_kernel<uint16_t>, grid_for_warps(n), CTA_THREADS, 0, items, n, kind, out, out2, out64);
  API_END();
}
int tb_motion_estimate_batch(const tb_me_item_t *items, int n, const int16_t *cand, int sample_bytes, int bitdepth, int speed, int bip, int fw, int fh,
                             tb_me_result_t *out) {
  API_BEGIN();
  if (sample_bytes != 1 && sample_bytes != 2) { set_err("tb_motion_estimate_batch: sample_bytes must be 1 or 2", cudaSuccess); return TB_ERR_ARG; }
  if (n <= 0) return TB_OK;
  // stream-ordered scratch: the sorted item list and the scheduler's counters (see me_batch_kernel)
  int *meta = nullptr, *idx = nullptr;
  CKB(cudaMallocAsync((void **)&meta, 128 * sizeof(int) + (size_t)n * sizeof(int), g.stream), "me scratch");
  idx = meta + 128;
  CKB(cudaMemsetAsync(meta, 0, 128 * sizeof(int), g.stream), "me scratch");
  const int sgrid = std::min((n + 255) / 256, g.sm_count * 8);
  const MeClassOf cls{speed, (sample_bytes == 1 && speed == 0) ? 1 : 0};
  LAUNCH((sched_hist_kernel<tb_me_item_t, MeClassOf>), sgrid, 256, 0, items, n, cls, meta);
  LAUNCH(sched_scan_kernel, 1, 32, 0, meta);
  LAUNCH((sched_scatter_kernel<tb_me_item_t, MeClassOf>), sgrid, 256, 0, items, n, cls, meta, idx);
  const int grid = std::min((n + WARPS_PER_CTA - 1) / WARPS_PER_CTA, g.sm_count * ME_MINBLOCKS);  // persistent: every CTA resident
  if (sample_bytes == 1) LAUNCH(me_batch_kernel<uint8_t>, grid, CTA_THREADS, 0, items, n, idx, meta, cand, bitdepth, speed, bip, fw, fh, out, g.me_stats);
  else LAUNCH(me_batch_kernel<uint16_t>, grid, CTA_THREADS, 0, items, n, idx, meta, cand, bitdepth, speed, bip, fw, fh, out, g.me_stats);
  CKB(cudaFreeAsync(meta, g.stream), "me scratch");
  API_END();
}
int tb_motion_estimate_bi_batch(const tb_me_bi_item_t *items, int n, const int16_t *cand, int sample_bytes, int bitdepth, int bip, int fw, int fh, tb_me_result_t *out) {
  API_BEGIN();
  if (sample_bytes != 1 && sample_bytes != 2) { set_err("tb_motion_estimate_bi_batch: sample_bytes must be 1 or 2", cudaSuccess); return TB_ERR_ARG; }
  if (n <= 0) return TB_OK;
  if (sample_bytes == 1) LAUNCH(me_bi_batch_kernel<uint8_t>, grid_for_warps(n), CTA_THREADS, 0, items, n, cand, bitdepth, bip, fw, fh, out);
  else LAUNCH(me_bi_batch_kernel<uint16_t>, grid_for_warps(n), CTA_THREADS, 0, items, n, cand, bitdepth, bip, fw, fh, out);
  API_END();
}
int tb_block_combine_batch(const tb_combine_item_t *items, int n, int sample_bytes, int op, int bitdepth) {
  API_BEGIN();
  if (n <= 0) return TB_OK;
  if (op < 0 || op > 2) return TB_ERR_ARG;
  if (sample_bytes == 1) LAUNCH(combine_batch_kernel<uint8_t>, grid_for_warps(n), CTA_THREADS, 0, items, n, op, bitdepth);
  else LAUNCH(combine_batch_kernel<uint16_t>, grid_for_warps(n), CTA_THREADS, 0, items, n, op, bitdepth);
  API_END();
}
int tb_me_set_stats(uint64_t *stats_dev) {
  g.me_stats = (unsigned long long *)stats_dev;
  return TB_OK;
}
int tb_interp_batch(const tb_interp_item_t *items, int n, int sample_bytes, int bitdepth, int bipred) {
  API_BEGIN();
  if (sample_bytes != 1 && sample_bytes != 2) { set_err("tb_interp_batch: sample_bytes must be 1 or 2", cudaSuccess); return TB_ERR_ARG; }
  if (n <= 0) return TB_OK;
  if (sample_bytes == 1) LAUNCH(interp_batch_kernel<uint8_t>, grid_for_warps((n + 3) / 4), CTA_THREADS, 0, items, n, bitdepth, bipred);
  else LAUNCH(interp_batch_kernel<uint16_t>, grid_for_warps((n + 3) / 4), CTA_THREADS, 0, items, n, bitdepth, bipred);
  API_END();
}
int tb_txfm_chain_batch(const tb_txfm_item_t *items, int n, int sample_bytes, int bitdepth, tb_txfm_result_t *out) {
  API_BEGIN();
  if (sample_bytes != 1 && sample_bytes != 2) { set_err("tb_txfm_chain_batch: sample_bytes must be 1 or 2", cudaSuccess); return TB_ERR_ARG; }
  if (n <= 0) return TB_OK;
  size_t smem = TX_TABLE_BYTES + sizeof(TxScratch) * WARPS_PER_CTA;
  int *meta = nullptr, *idx = nullptr;
  CKB(cudaMallocAsync((void **)&meta, 128 * sizeof(int) + (size_t)n * sizeof(int), g.stream), "txfm scratch");
  idx = meta + 128;
  CKB(cudaMemsetAsync(meta, 0, 128 * sizeof(int), g.stream), "txfm scratch");
  const int sgrid = std::min((n + 255) / 256, g.sm_count * 8);
  const TxClassOf cls{};
  LAUNCH((sched_hist_kernel<tb_txfm_item_t, TxClassOf>), sgrid, 256, 0, items, n, cls, meta);
  LAUNCH(sched_scan_kernel, 1, 32, 0, meta);
  LAUNCH((sched_scatter_kernel<tb_txfm_item_t, TxClassOf>), sgrid, 256, 0, items, n, cls, meta, idx);
  const int grid = std::min((n + 31) / 32, g.sm_count * TX_MINBLOCKS);  // persistent: every CTA resident
  if (sample_bytes == 1) LAUNCH(txfm_chain_kernel<uint8_t>, grid, CTA_THREADS, smem, items, n, idx, meta, bitdepth, out);
  else LAUNCH(txfm_chain_kernel<uint16_t>, grid, CTA_THREADS, smem, items, n, idx, meta, bitdepth, out);
  CKB(cudaFreeAsync(meta, g.stream), "txfm scratch");
  API_END();
}
int tb_intra_batch(const tb_intra_item_t *items, int n, int sample_bytes, int bitdepth) {
  API_BEGIN();
  if (sample_bytes != 1 && sample_bytes != 2) { set_err("tb_intra_batch: sample_bytes must be 1 or 2", cudaSuccess); return TB_ERR_ARG; }
  if (n <= 0) return TB_OK;
  if (sample_bytes == 1) LAUNCH(intra_batch_kernel<uint8_t>, grid_for_warps(n), CTA_THREADS, sizeof(IntraShared<uint8_t>) * WARPS_PER_CTA, items, n, bitdepth);
  else LAUNCH(intra_batch_kernel<uint16_t>, grid_for_warps(n), CTA_THREADS, sizeof(IntraShared<uint16_t>) * WARPS_PER_CTA, items, n, bitdepth);
  API_END();
}

// ---------------------------------------------------------------------------------------------------------------
// frame-level filters
// ---------------------------------------------------------------------------------------------------------------
int tb_deblock_frame(tb_frame_t *rec, const tb_blkinfo_t *bi, int qp, int bitdepth) {
  API_BEGIN();
  if (qp < 0 || qp > 51) return TB_ERR_ARG;
  if (rec->esz == 1) deblock_t<uint8_t>(rec, bi, qp, bitdepth);
  else deblock_t<uint16_t>(rec, bi, qp, bitdepth);
  API_END();
}

int tb_clpf_frame(tb_frame_t *rec, tb_frame_t *scratch, const tb_blkinfo_t *bi, const uint8_t *fb_on, int fb_size_log2, int strength, int bitdepth, int plane,
                  int qp) {
  API_BEGIN();
  if (!same_geometry(rec, scratch) || plane > 2) return TB_ERR_ARG;
  for (int p = (plane < 0 ? 0 : plane); p <= (plane < 0 ? 2 : plane); p++) {
    int fbl = p ? 4 : fb_size_log2;  // chroma always uses 16x16 filter blocks without signalling (enc/encode_frame.c:810-813)
    if (plane >= 0) fbl = fb_size_log2;
    if (rec->esz == 1) clpf_t<uint8_t>(rec, scratch, bi, fb_on, fbl, strength, bitdepth, p, qp);
    else clpf_t<uint16_t>(rec, scratch, bi, fb_on, fbl, strength, bitdepth, p, qp);
  }
  API_END();
}
int tb_clpf_detect_frame(const tb_frame_t *rec, const tb_frame_t *org, const tb_blkinfo_t *bi, int plane, int bitdepth, int qp, int32_t *sums) {
  API_BEGIN();
  if (plane < 0 || plane > 2) return TB_ERR_ARG;
  const int sub = plane ? 1 : 0, pw = rec->pw[plane], ph = rec->ph[plane], nb = (pw >> 3) * (ph >> 3);
  const int damping = bitdepth - 4 - (plane != 0) + (qp >> 4);
  if (rec->esz == 1)
    LAUNCH(clpf_detect_kernel<uint8_t>, grid_for_warps(nb), CTA_THREADS, 0, (const uint8_t *)rec->origin[plane], (const uint8_t *)org->origin[plane],
           rec->stride[plane], org->stride[plane], pw, ph, bi, rec->width >> 2, sub, bitdepth - 8, damping, sums);
  else
    LAUNCH(clpf_detect_kernel<uint16_t>, grid_for_warps(nb), CTA_THREADS, 0, (const uint16_t *)rec->origin[plane], (const uint16_t *)org->origin[plane],
           rec->stride[plane], org->stride[plane], pw, ph, bi, rec->width >> 2, sub, bitdepth - 8, damping, sums);
  API_END();
}

int tb_cdef_frame(tb_frame_t *rec, tb_frame_t *scratch, const tb_blkinfo_t *bi, const int8_t *fb_pri, const int8_t *fb_sec, int pri_damping, int sec_damping,
                  int32_t *dirvar, int bitdepth, int plane) {
  API_BEGIN();
  if (!same_geometry(rec, scratch) || plane < 0 || plane > 2) return TB_ERR_ARG;
  if (rec->esz == 1) cdef_t<uint8_t>(rec, scratch, bi, fb_pri, fb_sec, pri_damping, sec_damping, dirvar, bitdepth, plane);
  else cdef_t<uint16_t>(rec, scratch, bi, fb_pri, fb_sec, pri_damping, sec_damping, dirvar, bitdepth, plane);
  API_END();
}

int tb_cdef_search_mse(const tb_frame_t *rec, const tb_frame_t *org, const tb_blkinfo_t *blkinfo_dev, int speed, int pri_damping, int bitdepth, int32_t *dirvar_dev,
                       uint8_t *allskip_dev, uint64_t *mse_dev) {
  API_BEGIN();
  if (!same_geometry(rec, org) || speed < 0 || speed > 2) return TB_ERR_ARG;
  if (rec->esz == 1) cdef_search_t<uint8_t>(rec, org, blkinfo_dev, speed, pri_damping, bitdepth, dirvar_dev, allskip_dev, mse_dev);
  else cdef_search_t<uint16_t>(rec, org, blkinfo_dev, speed, pri_damping, bitdepth, dirvar_dev, allskip_dev, mse_dev);
  API_END();
}
int tb_pad_frame(tb_frame_t *f) {
  API_BEGIN();
  if (f->esz == 1) pad_t<uint8_t>(f, f, 1);
  else pad_t<uint16_t>(f, f, 1);
  API_END();
}
int tb_create_reference_frame(tb_frame_t *ref, const tb_frame_t *rec) {
  API_BEGIN();
  if (ref->width != rec->width || ref->height != rec->height || ref->esz != rec->esz) return TB_ERR_ARG;
  if (ref->esz == 1) pad_t<uint8_t>(ref, rec, 0);
  else pad_t<uint16_t>(ref, rec, 0);
  API_END();
}
int tb_scale_down2x2(const tb_frame_t *in, tb_frame_t *out) {
  API_BEGIN();
  if (out->width != in->width / 2 || out->height != in->height / 2 || in->esz != out->esz) return TB_ERR_ARG;
  dim3 blk(32, 8), grd((out->width + 31) / 32, (out->height + 7) / 8);
  if (in->esz == 1)
    LAUNCH(scale_down_kernel<uint8_t>, grd, blk, 0, (const uint8_t *)in->origin[0], in->stride[0], (uint8_t *)out->origin[0], out->stride[0], out->width,
           out->height);
  else
    LAUNCH(scale_down_kernel<uint16_t>, grd, blk, 0, (const uint16_t *)in->origin[0], in->stride[0], (uint16_t *)out->origin[0], out->stride[0], out->width,
           out->height);
  API_END();
}

}  // extern "C"

// ---- a21: temporal interpolation (common/temporal_interp.c:909-992) on resident frames
struct TiWork {
  int w = 0, h = 0, esz = 0, levels = 0;
  tb_frame *pyr[4][2] = {{nullptr}};
  short2 *mv0[4] = {nullptr}, *mv1[4] = {nullptr}, *sp0[4] = {nullptr}, *sp1[4] = {nullptr}, *m0[4] = {nullptr}, *m1[4] = {nullptr};
  int *progress = nullptr;
  int bw[4], bh[4];
};
static TiWork g_ti;

template <class S> static void ti_run(tb_frame *out, const tb_frame *r0, const tb_frame *r1, int ratio, int pos) {
  TiWork &W = g_ti;
  const int w = r0->width, h = r0->height, levels = W.levels;
  const int reversed = pos > ratio / 2, wt0 = reversed ? pos : ratio - pos, wt1 = ratio - wt0;
  const tb_frame *lv[4][2];
  lv[0][0] = r0; lv[0][1] = r1;
  for (int l = 1; l < levels; l++)
    for (int t = 0; t < 2; t++) {
      tb_frame *d = W.pyr[l][t];
      const tb_frame *s = lv[l - 1][t];
      dim3 blk(32, 8), grd((d->width + 31) / 32, (d->height + 7) / 8);
      LAUNCH(scale_down_kernel<S>, grd, blk, 0, (const S *)s->origin[0], s->stride[0], (S *)d->origin[0], d->stride[0], d->width, d->height);
      dim3 grd2((d->width + 2 * d->padh[0] + 31) / 32, (d->height + 2 * d->padv[0] + 7) / 8);
      LAUNCH(pad_copy_kernel<S>, grd2, blk, 0, (S *)d->origin[0], d->stride[0], (const S *)d->origin[0], d->stride[0], d->width, d->height, d->padh[0], d->padv[0], 1);
      lv[l][t] = d;
    }
  for (int l = levels - 1; l >= 0; l--) {
    TiLevel L;
    for (int t = 0; t < 2; t++) {
      const tb_frame *f = lv[l][reversed ? 1 - t : t];
      L.pic[t].y = f->origin[0]; L.pic[t].stride = f->stride[0]; L.pic[t].width = f->width; L.pic[t].height = f->height; L.pic[t].pad = f->padh[0];
    }
    L.mv0 = W.mv0[l]; L.mv1 = W.mv1[l]; L.bw = W.bw[l]; L.bh = W.bh[l]; L.wt0 = wt0; L.wt1 = wt1; L.reversed = reversed;
    L.guide = l != levels - 1 ? W.sp1[l] : nullptr; L.guide_reversed = reversed; L.guide_wt0 = wt0; L.progress = W.progress;
    const int nrows = L.bh / 2, n = L.bw * L.bh;
    ck(cudaMemsetAsync(W.progress, 0, sizeof(int) * (size_t)nrows, g.stream), "memset");
    if (!L.guide) {
      ck(cudaMemsetAsync(L.mv0, 0, sizeof(short2) * (size_t)n, g.stream), "memset");
      ck(cudaMemsetAsync(L.mv1, 0, sizeof(short2) * (size_t)n, g.stream), "memset");
    }
    LAUNCH(ti_me_kernel<S>, (nrows + 3) / 4, 128, 0, L);
    LAUNCH(ti_merge_kernel<S>, grid_for_warps(n), CTA_THREADS, 0, L, W.m0[l], W.m1[l]);
    if (l > 0)
      LAUNCH(ti_upscale_kernel, (W.bw[l - 1] * W.bh[l - 1] + 127) / 128, 128, 0, W.m1[l], W.bw[l], W.sp0[l - 1], W.sp1[l - 1], W.bw[l - 1], W.bh[l - 1], wt0, wt1);
  }
  const tb_frame *p0 = reversed ? r1 : r0, *p1 = reversed ? r0 : r1;
  for (int p = 0; p < 3; p++) {
    const int c = p ? 1 : 0, bs = c ? 4 : 8;
    dim3 blk(32, 8), grd((W.bw[0] * bs + 31) / 32, (W.bh[0] * bs + 7) / 8);
    LAUNCH(ti_interp_kernel<S>, grd, blk, 0, (const S *)p0->origin[p], p0->stride[p], (const S *)p1->origin[p], p1->stride[p], (S *)out->origin[p], out->stride[p], W.m0[0],
           W.m1[0], W.bw[0], W.bh[0], (w + 4) >> c, (h + 4) >> c, 4 >> c, c, wt0, wt1);
  }
}

extern "C" {

int tb_interpolate_frames(tb_frame_t *out, const tb_frame_t *ref0, const tb_frame_t *ref1, int ratio, int pos) {
  API_BEGIN();
  if (!same_geometry(ref0, ref1) || out->width != ref0->width || out->height != ref0->height || out->esz != ref0->esz || out->pad < 16) return TB_ERR_ARG;
  TiWork &W = g_ti;
  const int w = ref0->width, h = ref0->height;
  if (W.w != w || W.h != h || W.esz != ref0->esz) {  // (re)build the cached pyramid + vector fields for this geometry
    for (int l = 0; l < 4; l++) {
      for (int t = 0; t < 2; t++) if (W.pyr[l][t]) { tb_frame_destroy(W.pyr[l][t]); W.pyr[l][t] = nullptr; }
      short2 **arrs[6] = {&W.mv0[l], &W.mv1[l], &W.sp0[l], &W.sp1[l], &W.m0[l], &W.m1[l]};
      for (auto a : arrs) if (*a) { cudaFree(*a); *a = nullptr; }
    }
    if (W.progress) { cudaFree(W.progress); W.progress = nullptr; }
    // the reference derives the level count in double precision (common/temporal_interp.c:914)
    int levels = (int)(std::log10((double)(w < h ? w : h)) / std::log10(2.0) - 4.0);
    W.levels = levels < 4 ? levels : 4;
    if (W.levels < 1) return TB_ERR_ARG;
    for (int l = 0; l < W.levels; l++) {
      const int wl = w >> l, hl = h >> l;
      W.bw[l] = 2 * ((wl + 15) / 16); W.bh[l] = 2 * ((hl + 15) / 16);
      const size_t n = (size_t)W.bw[l] * W.bh[l] * sizeof(short2);
      short2 **arrs[6] = {&W.mv0[l], &W.mv1[l], &W.sp0[l], &W.sp1[l], &W.m0[l], &W.m1[l]};
      for (auto a : arrs) { if (cudaMalloc((void **)a, n) != cudaSuccess) return TB_ERR_CUDA; cudaMemsetAsync(*a, 0, n, g.stream); }
      if (l > 0)
        for (int t = 0; t < 2; t++)
          if (!(W.pyr[l][t] = tb_frame_create(wl & ~1 ? wl : 2, hl & ~1 ? hl : 2, 32, ref0->esz))) return TB_ERR_CUDA;
    }
    if (cudaMalloc((void **)&W.progress, sizeof(int) * (size_t)(W.bh[0] / 2 + 1)) != cudaSuccess) return TB_ERR_CUDA;
    W.w = w; W.h = h; W.esz = ref0->esz;
  }
  if (ref0->esz == 1) ti_run<uint8_t>(out, ref0, ref1, ratio, pos);
  else ti_run<uint16_t>(out, ref0, ref1, ratio, pos);
  API_END();
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// (A) drop-in symbols.  Each stages its host operands (slots 0..3), launches, copies results back, synchronises.
// ---------------------------------------------------------------------------------------------------------------
namespace {

template <class S> int sad_impl(const S *a, const S *b, int as, int bs, int w, int h, int kind, int *xout, uint64_t *ssd) {
  need_ctx("sad");
  const int lo = kind == 1 ? -3 : 0, hi = kind == 1 ? 3 : 0;
  Win wa = win(0, a, sizeof(S), as, 0, 0, w, h, true), wb = win(1, b, sizeof(S), bs, lo, 0, w + hi, h, true);
  struct Out { uint32_t s; int32_t x; uint64_t ssd; tb_sad_item_t it; };
  Out *d = (Out *)slot_buf(2, sizeof(Out));
  tb_sad_item_t it;
  it.a = wa.dev(); it.b = wb.dev(); it.astride = wa.dstride(); it.bstride = wb.dstride(); it.width = (uint16_t)w; it.height = (uint16_t)h; it.pad = 0;
  ck(cudaMemcpyAsync(&d->it, &it, sizeof(it), cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(sad_batch_kernel<S>, 1, 32, 0, &d->it, 1, kind, &d->s, &d->x, &d->ssd);
  Out r;
  ck(cudaMemcpyAsync(&r, d, sizeof(uint32_t) + sizeof(int32_t) + sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
  if (xout) *xout = r.x;
  if (ssd) *ssd = r.ssd;
  return (int)r.s;
}

template <class S> unsigned fast_impl(const S *a, const S *b, int as, int bs, int w, int h, int which, int *x, int *y) {
  need_ctx("fast subpel sad");
  Win wa = win(0, a, sizeof(S), as, 0, 0, w, h, true), wb = win(1, b, sizeof(S), bs, -2, -2, w + 3, h + 3, true);
  int32_t *d = (int32_t *)slot_buf(2, 16);
  LAUNCH(fast_subpel_kernel<S>, 1, 32, 0, (const S *)wa.dev(), wa.dstride(), (const S *)wb.dev(), wb.dstride(), w, h, which, which ? *x : 0, which ? *y : 0, d);
  int32_t r[3];
  ck(cudaMemcpyAsync(r, d, sizeof(r), cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
  *x = r[1];
  *y = r[2];
  return (unsigned)r[0];
}

template <class S> void interp_impl(int w, int h, int xoff, int yoff, S *qp, int qs, const S *ip, int is, int chroma, int bipred, int bitdepth) {
  need_ctx("interp");
  const int lo = chroma ? -1 : -2, hi = chroma ? 2 : 3;
  Win wi = win(0, ip, sizeof(S), is, lo, lo, w + hi, h + hi, true), wo = win(1, qp, sizeof(S), qs, 0, 0, w, h, false);
  LAUNCH(interp_frac_kernel<S>, (w * h + 127) / 128, 128, 0, (S *)wo.dev(), wo.dstride(), (const S *)wi.dev(), wi.dstride(), w, h, xoff, yoff, chroma, bipred, bitdepth);
  win_download(wo, qp, 0, 0, w, h);
  sync();
}

template <class S> void clpf_impl(const S *src, S *dst, int ss, int ds, int x0, int y0, int sx, int sy, int bt, unsigned strength, unsigned dmp) {
  need_ctx("clpf_block");
  Win wi = win(0, src, sizeof(S), ss, x0 - (bt & 1 ? 0 : 2), y0 - (bt & 4 ? 0 : 2), x0 + sx + (bt & 2 ? 0 : 2), y0 + sy + (bt & 8 ? 0 : 2), true);
  Win wo = win(1, dst, sizeof(S), ds, x0, y0, x0 + sx, y0 + sy, false);
  LAUNCH(clpf_block_kernel<S>, 1, 64, 0, (const S *)wi.dev(), (S *)wo.dev(), wi.dstride(), wo.dstride(), x0, y0, sx, sy, bt, (int)strength, (int)dmp);
  win_download(wo, dst, x0, y0, x0 + sx, y0 + sy);
  sync();
}

template <class S>
void detect_impl(const S *rec, const S *org, int x0, int y0, int width, int height, int so, int stride, unsigned strength, unsigned shift, unsigned size, unsigned dmp,
                 int multi, uint32_t res[4]) {
  need_ctx("detect_clpf");
  const int s = (int)size;
  Win wr = win(0, rec, sizeof(S), stride, max(0, x0 - 2), max(0, y0 - 2), min(width, x0 + s + 2), min(height, y0 + s + 2), true);
  Win wo = win(1, org, sizeof(S), so, x0, y0, x0 + s, y0 + s, true);
  uint32_t *d = (uint32_t *)slot_buf(2, 16);
  LAUNCH(clpf_detect_block_kernel<S>, 1, 32, 0, (const S *)wr.dev(), (const S *)wo.dev(), x0, y0, width, height, wo.dstride(), wr.dstride(), (int)strength, (int)shift, s,
         (int)dmp, multi, d);
  ck(cudaMemcpyAsync(res, d, 16, cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
}

template <class S> void block_avg_impl(S *p, const S *r0, const S *r1, int sp, int s0, int s1, int w, int h) {
  need_ctx("block_avg");
  Win a = win(0, r0, sizeof(S), s0, 0, 0, w, h, true), b = win(1, r1, sizeof(S), s1, 0, 0, w, h, true), o = win(2, p, sizeof(S), sp, 0, 0, w, h, false);
  LAUNCH(block_avg_kernel<S>, (w * h + 127) / 128, 128, 0, (S *)o.dev(), o.dstride(), (const S *)a.dev(), a.dstride(), (const S *)b.dev(), b.dstride(), w, h);
  win_download(o, p, 0, 0, w, h);
  sync();
}

template <class S> void scale_impl(tb_yuv_frame *sin, tb_yuv_frame *sout) {
  need_ctx("scale_frame_down2x2");
  const int wo = sout->width, ho = sout->height;
  Win i = win(0, sin->y, sizeof(S), sin->stride_y, 0, 0, 2 * wo, 2 * ho, true), o = win(1, sout->y, sizeof(S), sout->stride_y, 0, 0, wo, ho, false);
  dim3 blk(32, 8), grd((wo + 31) / 32, (ho + 7) / 8);
  LAUNCH(scale_down_kernel<S>, grd, blk, 0, (const S *)i.dev(), i.dstride(), (S *)o.dev(), o.dstride(), wo, ho);
  win_download(o, sout->y, 0, 0, wo, ho);
  sync();
}

template <class S> int cdef_dir_impl(const S *img, int stride, int32_t *var, int coeff_shift) {
  need_ctx("cdef_find_dir");
  Win i = win(0, img, sizeof(S), stride, 0, 0, 8, 8, true);
  int32_t *d = (int32_t *)slot_buf(2, 8);
  LAUNCH(cdef_dir_block_kernel<S>, 1, 32, 0, (const S *)i.dev(), i.dstride(), coeff_shift, d);
  int32_t r[2];
  ck(cudaMemcpyAsync(r, d, 8, cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
  *var = r[1];
  return r[0];
}

}  // namespace

extern "C" {

#define TB_DEF_SAMPLE_SYMBOLS(S, SFX)                                                                                                               \
  int sad_calc_simd_##SFX(S *a, S *b, int as, int bs, int w, int h) { return sad_impl<S>(a, b, as, bs, w, h, 0, nullptr, nullptr); }               \
  int sad_calc_simd_unaligned_##SFX(S *a, S *b, int as, int bs, int w, int h) { return sad_impl<S>(a, b, as, bs, w, h, 0, nullptr, nullptr); }     \
  uint64_t ssd_calc_simd_##SFX(S *a, S *b, int as, int bs, int size) {                                                                             \
    uint64_t v = 0;                                                                                                                                 \
    sad_impl<S>(a, b, as, bs, size, size, 2, nullptr, &v);                                                                                          \
    return v;                                                                                                                                       \
  }                                                                                                                                                 \
  unsigned int widesad_calc_simd_##SFX(S *a, S *b, int as, int bs, int w, int h, int *x) { return (unsigned)sad_impl<S>(a, b, as, bs, w, h, 1, x, nullptr); } \
  unsigned int sad_calc_fasthalf_simd_##SFX(const S *a, const S *b, int as, int bs, int w, int h, int *x, int *y) {                                \
    return fast_impl<S>(a, b, as, bs, w, h, 0, x, y);                                                                                               \
  }                                                                                                                                                 \
  unsigned int sad_calc_fastquarter_simd_##SFX(const S *o, const S *r, int os, int rs, int w, int h, int *x, int *y) {                             \
    return fast_impl<S>(o, r, os, rs, w, h, 1, x, y);                                                                                               \
  }                                                                                                                                                 \
  /* the reference adds the C sums and then the SIMD sums: both accumulators grow by twice the block sums (enc/enc_kernels.c:257-294) */            \
  void detect_clpf_simd_##SFX(const S *rec, const S *org, int x0, int y0, int width, int height, int so, int stride, int *sum0, int *sum1,         \
                              unsigned int strength, unsigned int shift, unsigned int size, unsigned int dmp) {                                     \
    uint32_t r[4];                                                                                                                                  \
    detect_impl<S>(rec, org, x0, y0, width, height, so, stride, strength, shift, size, dmp, 0, r);                                                  \
    *sum0 += 2 * (int)(r[0] >> (shift * 2));                                                                                                        \
    *sum1 += 2 * (int)(r[1] >> (shift * 2));                                                                                                        \
  }                                                                                                                                                 \
  void detect_multi_clpf_simd_##SFX(const S *rec, const S *org, int x0, int y0, int width, int height, int so, int stride, int *sum,               \
                                    unsigned int shift, unsigned int size, unsigned int dmp) {                                                      \
    uint32_t r[4];                                                                                                                                  \
    detect_impl<S>(rec, org, x0, y0, width, height, so, stride, 0, shift, size, dmp, 1, r);                                                         \
    for (int t = 0; t < 4; t++) sum[t] += (int)(r[t] >> (shift * 2));                                                                               \
  }                                                                                                                                                 \
  void block_avg_simd_##SFX(S *p, S *r0, S *r1, int sp, int s0, int s1, int w, int h) { block_avg_impl<S>(p, r0, r1, sp, s0, s1, w, h); }           \
  void get_inter_prediction_luma_simd_##SFX(int w, int h, int xoff, int yoff, S *qp, int qs, const S *ip, int is, int bipred, int bitdepth) {      \
    interp_impl<S>(w, h, xoff, yoff, qp, qs, ip, is, 0, bipred, bitdepth);                                                                          \
  }                                                                                                                                                 \
  void get_inter_prediction_chroma_simd_##SFX(int w, int h, int xoff, int yoff, S *qp, int qs, const S *ip, int is, int bitdepth) {                \
    interp_impl<S>(w, h, xoff, yoff, qp, qs, ip, is, 1, 0, bitdepth);                                                                               \
  }                                                                                                                                                 \
  void clpf_block4_##SFX(const S *src, S *dst, int ss, int ds, int x0, int y0, int sizey, int bt, unsigned int strength, unsigned int dmp) {       \
    clpf_impl<S>(src, dst, ss, ds, x0, y0, 4, sizey, bt, strength, dmp);                                                                            \
  }                                                                                                                                                 \
  void clpf_block8_##SFX(const S *src, S *dst, int ss, int ds, int x0, int y0, int sizey, int bt, unsigned int strength, unsigned int dmp) {       \
    clpf_impl<S>(src, dst, ss, ds, x0, y0, 8, sizey, bt, strength, dmp);                                                                            \
  }                                                                                                                                                 \
  void clpf_block4_noclip_##SFX(const S *src, S *dst, int ss, int ds, int x0, int y0, int sizey, unsigned int strength, unsigned int dmp) {        \
    clpf_impl<S>(src, dst, ss, ds, x0, y0, 4, sizey, 0, strength, dmp);                                                                             \
  }                                                                                                                                                 \
  void clpf_block8_noclip_##SFX(const S *src, S *dst, int ss, int ds, int x0, int y0, int sizey, unsigned int strength, unsigned int dmp) {        \
    clpf_impl<S>(src, dst, ss, ds, x0, y0, 8, sizey, 0, strength, dmp);                                                                             \
  }                                                                                                                                                 \
  void scale_frame_down2x2_simd_##SFX(struct tb_yuv_frame *sin, struct tb_yuv_frame *sout) { scale_impl<S>(sin, sout); }                            \
  int cdef_find_dir_simd_##SFX(const S *img, int stride, int32_t *var, int coeff_shift) { return cdef_dir_impl<S>(img, stride, var, coeff_shift); }

TB_DEF_SAMPLE_SYMBOLS(uint8_t, lbd)
TB_DEF_SAMPLE_SYMBOLS(uint16_t, hbd)

void transform_simd(const int16_t *block, int16_t *coeff, int size, int fast, int bitdepth) {
  need_ctx("transform");
  const int q = size < 16 ? size : 16;
  int16_t *din = (int16_t *)slot_buf(3, (size_t)size * size * 2), *dout = (int16_t *)slot_buf(2, (size_t)size * size * 2);
  ck(cudaMemcpyAsync(din, block, (size_t)size * size * 2, cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(fwd_transform_kernel, 1, 32, 0, din, dout, size, fast, bitdepth);
  // only the low min(size,16)^2 coefficients are produced (common/transform.c:289-307); the rest of coeff[] is untouched
  ck(cudaMemcpy2DAsync(coeff, (size_t)size * 2, dout, (size_t)size * 2, (size_t)q * 2, q, cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
}
void inverse_transform_simd(const int16_t *coeff, int16_t *block, int size, int bitdepth) {
  need_ctx("inverse_transform");
  const int q = size < 16 ? size : 16;
  int16_t *din = (int16_t *)slot_buf(3, (size_t)size * size * 2), *dout = (int16_t *)slot_buf(2, (size_t)size * size * 2);
  ck(cudaMemcpy2DAsync(din, (size_t)size * 2, coeff, (size_t)size * 2, (size_t)q * 2, q, cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(inv_transform_kernel, 1, 32, 0, din, dout, size, bitdepth);
  ck(cudaMemcpyAsync(block, dout, (size_t)size * size * 2, cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
}
int check_nz_area(const int16_t *coeff, int size) {
  need_ctx("check_nz_area");
  const int q = size < 16 ? size : 16;
  int16_t *din = (int16_t *)slot_buf(3, (size_t)size * size * 2);
  int32_t *d = (int32_t *)slot_buf(2, 8);
  ck(cudaMemcpy2DAsync(din, (size_t)size * 2, coeff, (size_t)size * 2, (size_t)q * 2, q, cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(check_nz_kernel, 1, 32, 0, din, size, d);
  return fetch<int32_t>(d);
}
int calc_cbp_simd(int16_t *block, int size, int threshold) {
  need_ctx("calc_cbp");
  int16_t *din = (int16_t *)slot_buf(3, (size_t)size * size * 2);
  int32_t *d = (int32_t *)slot_buf(2, 8);
  ck(cudaMemcpyAsync(din, block, (size_t)size * size * 2, cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(calc_cbp_kernel, 1, 32, 0, din, size, threshold, d);
  return fetch<int32_t>(d);
}
void cdef_filter_block_simd(uint8_t *dst8, uint16_t *dst16, int dstride, const uint16_t *in, int sstride, int pri_strength, int sec_strength, int dir,
                            int pri_damping, int sec_damping, int bsize, int cdef_directions[8][2], int coeff_shift) {
  (void)cdef_directions;  // offsets are re-derived from (dy,dx) and the staged pitch; callers build the table with cdef_init()
  need_ctx("cdef_filter_block");
  Win i = win(0, in, 2, sstride, -2, -2, bsize + 2, bsize + 2, true);
  const int esz = dst8 ? 1 : 2;
  void *hd = dst8 ? (void *)dst8 : (void *)dst16;
  Win o = win(1, hd, esz, dstride, 0, 0, bsize, bsize, false);
  LAUNCH(cdef_block_kernel, 1, 64, 0, dst8 ? (uint8_t *)o.dev() : nullptr, dst8 ? nullptr : (uint16_t *)o.dev(), o.dstride(), (const uint16_t *)i.dev(), i.dstride(),
         pri_strength, sec_strength, dir, pri_damping, sec_damping, bsize, coeff_shift);
  win_download(o, hd, 0, 0, bsize, bsize);
  sync();
}

// single-block, host-buffer forms of host-object functions on the path (not reference exports; used by parity tests
// and by hosts that have not been batched yet)
int tb_quantize(const int16_t *coeff, int16_t *coeffq, int qp, int size, int coeff_block_type) { /* enc/encode_block.c:84 */
  need_ctx("quantize");
  const int q = size < 16 ? size : 16;
  int16_t *din = (int16_t *)slot_buf(3, (size_t)size * size * 2), *dout = (int16_t *)slot_buf(2, 512 + 16);
  ck(cudaMemcpy2DAsync(din, (size_t)size * 2, coeff, (size_t)size * 2, (size_t)q * 2, q, cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(quant_kernel, 1, 32, 0, din, dout, qp, size, coeff_block_type, (int32_t *)(dout + 256));
  ck(cudaMemcpyAsync(coeffq, dout, (size_t)q * q * 2, cudaMemcpyDeviceToHost, g.stream), "D2H");
  return fetch<int32_t>(dout + 256);
}
void tb_dequantize(const int16_t *coeffq, int16_t *rcoeff, int qp, int size) { /* common/common_block.c:45 */
  need_ctx("dequantize");
  const int q = size < 16 ? size : 16;
  int16_t *din = (int16_t *)slot_buf(3, 512), *dout = (int16_t *)slot_buf(2, (size_t)size * size * 2);
  ck(cudaMemcpyAsync(din, coeffq, (size_t)q * q * 2, cudaMemcpyHostToDevice, g.stream), "H2D");
  LAUNCH(dequant_kernel, 1, 32, 0, din, dout, qp, size);
  ck(cudaMemcpy2DAsync(rcoeff, (size_t)size * 2, dout, (size_t)size * 2, (size_t)q * 2, q, cudaMemcpyDeviceToHost, g.stream), "D2H");
  sync();
}
/* common/common_block.c:347 (4:2:0): y = n*n luma prediction (pitch n), u/v = (n/2)^2 chroma predictions (pitch cstride/2), ry = reconstructed luma */
void tb_improve_uv_prediction(int sample_bytes, const void *y, void *u, void *v, const void *ry, int n, int cstride, int stride, int sub, int bitdepth) {
  need_ctx("improve_uv_prediction");
  const int nc = n >> sub, cs = cstride >> sub;
  Win wy = win(0, y, sample_bytes, n, 0, 0, n, n, true), wr = win(1, ry, sample_bytes, stride, 0, 0, n, n, true);
  Win wu = win(2, u, sample_bytes, cs, 0, 0, nc, nc, true), wv = win(3, v, sample_bytes, cs, 0, 0, nc, nc, true);
  // the kernel derives the chroma pitch as cstride >> sub and the luma-prediction pitch as n: restage compactly
  if (wy.dstride() != n || wu.dstride() != cs) {
    // staged pitches are padded to 16 bytes; use compact copies for y, u, v instead
    char *cy = (char *)slot_buf(4, (size_t)n * n * sample_bytes), *cu = (char *)slot_buf(5, (size_t)nc * cs * sample_bytes + 64),
         *cv = (char *)slot_buf(6, (size_t)nc * cs * sample_bytes + 64);
    ck(cudaMemcpyAsync(cy, y, (size_t)n * n * sample_bytes, cudaMemcpyHostToDevice, g.stream), "H2D");
    ck(cudaMemcpy2DAsync(cu, (size_t)cs * sample_bytes, u, (size_t)cs * sample_bytes, (size_t)nc * sample_bytes, nc, cudaMemcpyHostToDevice, g.stream), "H2D");
    ck(cudaMemcpy2DAsync(cv, (size_t)cs * sample_bytes, v, (size_t)cs * sample_bytes, (size_t)nc * sample_bytes, nc, cudaMemcpyHostToDevice, g.stream), "H2D");
    if (sample_bytes == 1) LAUNCH(cfl_kernel<uint8_t>, 1, 32, 0, (const uint8_t *)cy, (uint8_t *)cu, (uint8_t *)cv, (const uint8_t *)wr.dev(), n, cstride, wr.dstride(), sub, bitdepth);
    else LAUNCH(cfl_kernel<uint16_t>, 1, 32, 0, (const uint16_t *)cy, (uint16_t *)cu, (uint16_t *)cv, (const uint16_t *)wr.dev(), n, cstride, wr.dstride(), sub, bitdepth);
    ck(cudaMemcpy2DAsync(u, (size_t)cs * sample_bytes, cu, (size_t)cs * sample_bytes, (size_t)nc * sample_bytes, nc, cudaMemcpyDeviceToHost, g.stream), "D2H");
    ck(cudaMemcpy2DAsync(v, (size_t)cs * sample_bytes, cv, (size_t)cs * sample_bytes, (size_t)nc * sample_bytes, nc, cudaMemcpyDeviceToHost, g.stream), "D2H");
    sync();
    return;
  }
  if (sample_bytes == 1) LAUNCH(cfl_kernel<uint8_t>, 1, 32, 0, (const uint8_t *)wy.dev(), (uint8_t *)wu.dev(), (uint8_t *)wv.dev(), (const uint8_t *)wr.dev(), n, cstride, wr.dstride(), sub, bitdepth);
  else LAUNCH(cfl_kernel<uint16_t>, 1, 32, 0, (const uint16_t *)wy.dev(), (uint16_t *)wu.dev(), (uint16_t *)wv.dev(), (const uint16_t *)wr.dev(), n, cstride, wr.dstride(), sub, bitdepth);
  win_download(wu, u, 0, 0, nc, nc);
  win_download(wv, v, 0, 0, nc, nc);
  sync();
}

// read-only tap tables referenced by common/inter_prediction.c:47-49 (values: common/common_kernels.c:1905-1928)
#define TB_TAPS(SFX)                                                                                                                                 \
  extern const int16_t coeffs_standard_##SFX[4][8] = {{0, 0, 64, 0, 0, 0, 0, 0}, {1, -7, 55, 19, -5, 1, 0, 0}, {1, -7, 38, 38, -7, 1, 0, 0}, {1, -5, 19, 55, -7, 1, 0, 0}}; \
  extern const int16_t coeffs_bipred_##SFX[4][8] = {{0, 0, 64, 0, 0, 0, 0, 0}, {2, -10, 59, 17, -5, 1, 0, 0}, {1, -8, 39, 39, -8, 1, 0, 0}, {1, -5, 17, 59, -10, 2, 0, 0}};  \
  extern const int16_t coeffs_chroma_##SFX[8][4] = {{0, 64, 0, 0}, {-2, 58, 10, -2}, {-4, 54, 16, -2}, {-4, 44, 28, -4}, {-4, 36, 36, -4}, {-4, 28, 44, -4}, {-2, 16, 54, -4}, {-2, 10, 58, -2}};
TB_TAPS(lbd)
TB_TAPS(hbd)

}  // extern "C"
