// wrcu_api.cu — the C ABI of include/wrcu.h: context, textures, per-frame
// tables, target binding, clears and the draw dispatch.  Host side of the
// B200 backend; every pixel is produced by the CUDA kernels in raster.cuh /
// setup_*.cuh.  There is no CPU rasterisation path in this library.
#include <stdarg.h>
#include <stdlib.h>
#include <vector>

#include "raster.cuh"
#include "shader_clip_rect.cuh"
#include "shader_quad_mask.cuh"
#include "shader_image.cuh"
#include "shader_text.cuh"
#include "shader_gradient.cuh"
#include "shader_box_shadow.cuh"
#include "shader_composite.cuh"
#include "shader_composite_yuv.cuh"
#include "blit_yuv.cuh"
#include "shader_opacity.cuh"
#include "shader_blend.cuh"
#include "shader_mix_blend.cuh"
#include "shader_blur.cuh"
#include "shader_scale.cuh"
#include "shader_cs_gradient.cuh"
#include "shader_border.cuh"
#include "setup_brush.cuh"
#include "setup_clip.cuh"
#include "setup_quad.cuh"
#include "wrcu_internal.h"

int wrcu_fail(wrcu_ctx* c, int code, const char* fmt, ...) {
  if (c) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(c->err, sizeof c->err, fmt, ap);
    va_end(ap);
    if (!c->sticky_error) c->sticky_error = code;
  }
  return code;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- deferred submission ---------------------------------------------------------------------------
// wrcu_clear / wrcu_draw_batch queue their work; flush_pending runs the queue: one H2D copy of everything
// staged since the last flush (tables, instances, the job table), ONE set-up launch over all queued batches
// (wr_setup_multi), then the clears and raster launches in submission order.  A page is ~150 batches of a
// few instances: with a launch pair per batch its frame time was 150 x the ~10 us latency chain of a set-up
// kernel; now that chain is paid once.  Everything else in the ABI flushes first, so callers see the same
// ordering as before.
struct PendingOp {
  int type = 0;                 // 0 = clear, 1 = batch
  // clear
  uint8_t* c_ptr = nullptr; int c_pitch = 0, c_fmt = 0; uint32_t c_val = 0;
  uint8_t* d_ptr = nullptr; int d_pitch = 0; uint32_t d_val = 0;
  int cx0 = 0, cy0 = 0, cx1 = 0, cy1 = 0;
  // batch
  int kind = 0, blend = 0, n = 0, sblocks = 0;
  uint32_t features = 0;
  unsigned grid_x = 0, grid_y = 0;
  size_t bin_need = 0, inst_off = 0, views_off = (size_t)-1;
  std::vector<const uint8_t*> tex_reads;  // wrcu_draw_composite_tiles: the instances' textures (stream scheduling)
  SetupArgs sa;
  RasterArgs ra;
};
static std::vector<PendingOp>& pending(wrcu_ctx* c) {
  if (!c->pending_ops) c->pending_ops = new std::vector<PendingOp>();
  return *(std::vector<PendingOp>*)c->pending_ops;
}

static int flush_pending(wrcu_ctx* c);

static int fmt_bpp(int fmt) {
  switch (fmt) {
    case WRCU_FMT_RGBA8: return 4;
    case WRCU_FMT_R8: return 1;
    case WRCU_FMT_RGBAF32: return 16;
    case WRCU_FMT_RGBAI32: return 16;
    case WRCU_FMT_DEPTH24: return 4;
    case WRCU_FMT_RG8: return 2;
    case WRCU_FMT_R16: return 2;
    case WRCU_FMT_RG16: return 4;
  }
  return 0;
}

// ---- launch helpers: real kernel launches, or (tests only) host loops -------------
#ifdef WRCU_HOSTEMU
#define WR_LAUNCH(kernel, grid, block, stream, ...) kernel(__VA_ARGS__)
#define WR_GLOBAL static
#else
#define WR_LAUNCH(kernel, grid, block, stream, ...) kernel<<<grid, block, 0, stream>>>(__VA_ARGS__)
#define WR_GLOBAL __global__
#endif
#ifdef WRCU_HOSTEMU
#define WR_LAUNCH_CHAIN(kernel, grid, block, ra) kernel(ra)
#else
#define WR_LAUNCH_CHAIN(kernel, grid, block, ra) wr_launch_chain(c, kernel, (unsigned)(grid), (unsigned)(block), 0, ra)
#endif

// ---- small kernels ---------------------------------------------------------------
WR_GLOBAL void wr_init_batch_info(BatchInfo* info, int n) {  // once, at context creation
#ifdef WRCU_HOSTEMU
  for (int i = 0; i < n; i++) wr_reset_batch_info(info + i);
#else
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) wr_reset_batch_info(info + i);
#endif
}

// Clear (swgl/src/gl.cc:2498-2518 → clear_buffer): fills a rect of a 4-byte or
// 1-byte target.  Rows are written as 16-byte vectors where alignment allows.
#ifdef WRCU_HOSTEMU
static void wr_clear_u32(uint8_t* base, int pitch, int x0, int y0, int x1, int y1, uint32_t v) {
  for (int y = y0; y < y1; y++) for (int x = x0; x < x1; x++) ((uint32_t*)(base + (size_t)y * pitch))[x] = v;
}
static void wr_clear_u8(uint8_t* base, int pitch, int x0, int y0, int x1, int y1, uint8_t v) {
  for (int y = y0; y < y1; y++) for (int x = x0; x < x1; x++) (base + (size_t)y * pitch)[x] = v;
}
#else
__global__ void wr_clear_u32(uint8_t* base, int pitch, int x0, int y0, int x1, int y1, uint32_t v) {
  int y = y0 + blockIdx.y;
  if (y >= y1) return;
  uint32_t* row = (uint32_t*)(base + (size_t)y * pitch);
  // vector body on 4-pixel boundaries
  int xa = (x0 + 3) & ~3, xb = x1 & ~3;
  if (xa >= xb) {
    for (int x = x0 + blockIdx.x * blockDim.x + threadIdx.x; x < x1; x += gridDim.x * blockDim.x) row[x] = v;
    return;
  }
  uint4 vv = make_uint4(v, v, v, v);
  for (int x = xa + 4 * (blockIdx.x * blockDim.x + threadIdx.x); x < xb; x += 4 * gridDim.x * blockDim.x)
    *(uint4*)(row + x) = vv;
  if (blockIdx.x == 0) {
    for (int x = x0 + threadIdx.x; x < xa; x += blockDim.x) row[x] = v;
    for (int x = xb + threadIdx.x; x < x1; x += blockDim.x) row[x] = v;
  }
}
__global__ void wr_clear_u8(uint8_t* base, int pitch, int x0, int y0, int x1, int y1, uint8_t v) {
  int y = y0 + blockIdx.y;
  if (y >= y1) return;
  uint8_t* row = base + (size_t)y * pitch;
  for (int x = x0 + blockIdx.x * blockDim.x + threadIdx.x; x < x1; x += gridDim.x * blockDim.x) row[x] = v;
}

#endif

// ---- update path kernels (SURVEY.md §8f rank 3) -------------------------------------------
struct UploadRectDev { int x, y, w, h; unsigned long long offset, stride; };
// Scatter staged rects into a texture: CTA (x = rect, y = row slice); a row is moved 16 bytes per
// thread where source and destination are both 16-byte aligned, bytewise otherwise.
WR_GLOBAL void wr_upload_scatter(uint8_t* dst, int pitch, int bpp, const UploadRectDev* rects, int n,
                                 const uint8_t* staging) {
#ifdef WRCU_HOSTEMU
  for (int i = 0; i < n; i++) {
    const UploadRectDev r = rects[i];
    for (int row = 0; row < r.h; row++)
      memcpy(dst + (size_t)(r.y + row) * pitch + (size_t)r.x * bpp, staging + r.offset + (size_t)row * r.stride,
             (size_t)r.w * bpp);
  }
#else
  const UploadRectDev r = rects[blockIdx.x];
  const size_t row_bytes = (size_t)r.w * bpp;
  for (int row = blockIdx.y; row < r.h; row += gridDim.y) {
    const uint8_t* s = staging + r.offset + (size_t)row * r.stride;
    uint8_t* d = dst + (size_t)(r.y + row) * pitch + (size_t)r.x * bpp;
    if ((((uintptr_t)s | (uintptr_t)d) & 15) == 0) {
      const size_t nv = row_bytes >> 4;
      for (size_t i = threadIdx.x; i < nv; i += blockDim.x) ((uint4*)d)[i] = __ldg((const uint4*)s + i);
      for (size_t i = (nv << 4) + threadIdx.x; i < row_bytes; i += blockDim.x) d[i] = s[i];
    } else if (bpp == 4 && (((uintptr_t)s | (uintptr_t)d) & 3) == 0) {
      for (size_t i = threadIdx.x; i < (size_t)r.w; i += blockDim.x) ((uint32_t*)d)[i] = __ldg((const uint32_t*)s + i);
    } else {
      for (size_t i = threadIdx.x; i < row_bytes; i += blockDim.x) d[i] = s[i];
    }
  }
#endif
}
struct GpuCacheCopyDev { unsigned block_index, block_count; unsigned short u, v; };
// GpuCacheUpdate::Copy: one warp per update, a 16-byte block per lane (gpu_cache_update.glsl
// draws one point per block).
WR_GLOBAL void wr_gpu_cache_scatter(float4* cache, int rows, const GpuCacheCopyDev* updates, int n,
                                    const float4* blocks, int n_blocks) {
#ifdef WRCU_HOSTEMU
  for (int i = 0; i < n; i++) {
    const GpuCacheCopyDev u = updates[i];
    for (unsigned b = 0; b < u.block_count; b++) {
      size_t dsti = (size_t)u.v * 1024 + u.u + b;
      if (u.v < rows && u.u + b < 1024 && u.block_index + b < (unsigned)n_blocks) cache[dsti] = blocks[u.block_index + b];
    }
  }
#else
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const GpuCacheCopyDev u = updates[warp];
  if (u.v >= rows) return;
  for (unsigned b = lane; b < u.block_count; b += 32)
    if (u.u + b < 1024 && u.block_index + b < (unsigned)n_blocks)
      cache[(size_t)u.v * 1024 + u.u + b] = __ldg(blocks + u.block_index + b);
#endif
}

// ---- context -----------------------------------------------------------------------
extern "C" int wrcu_abi_version(void) { return WRCU_ABI_VERSION; }

extern "C" const char* wrcu_get_string(int what) {
  switch (what) {
    case 0: return "Software WebRender";  // keeps is_software host behaviour (gl.cc:1214)
    case 1: return "wrcu: B200 (sm_100a) tile-resident CUDA rasteriser";
    default: return "";
  }
}

static int arena_init(wrcu_ctx* c, Arena* a, size_t cap) {
  a->cap = cap;
  a->used = 0;
  WRCU_CUDA(c, cudaMallocHost((void**)&a->host, cap));
  WRCU_CUDA(c, cudaMalloc((void**)&a->dev, cap));
  WRCU_CUDA(c, cudaEventCreateWithFlags(&a->done, cudaEventDisableTiming));
  return WRCU_OK;
}

extern "C" int wrcu_ctx_create(int device_ordinal, wrcu_ctx** out) {
  if (!out) return WRCU_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device_ordinal < 0 || device_ordinal >= n)
    return WRCU_ERR_NO_DEVICE;  // fail loudly: there is no CPU path
  if (cudaSetDevice(device_ordinal) != cudaSuccess) return WRCU_ERR_NO_DEVICE;
  wrcu_ctx* c = new wrcu_ctx();
  c->device = device_ordinal;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device_ordinal) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return WRCU_ERR_CUDA;
  }
  int rc;
  if ((rc = arena_init(c, &c->arena[0], 64u << 20)) != WRCU_OK ||
      (rc = arena_init(c, &c->arena[1], 64u << 20)) != WRCU_OK) {
    delete c;
    return rc;
  }
  cudaEventCreate(&c->t0);
  cudaEventCreate(&c->t1);
  cudaEventCreate(&c->p0);
  cudaEventCreate(&c->p1);
  if (cudaMalloc((void**)&c->batch_info, 2 * (size_t)wrcu_ctx::QMAX * sizeof(BatchInfo)) != cudaSuccess ||
      cudaMalloc((void**)&c->dev_err, sizeof(int)) != cudaSuccess ||
      cudaMalloc((void**)&c->pool_ctr, 4 * sizeof(int)) != cudaSuccess) {
    delete c;
    return WRCU_ERR_OOM;
  }
  cudaMemsetAsync(c->dev_err, 0, sizeof(int), c->stream);
  cudaMemsetAsync(c->pool_ctr, 0, 4 * sizeof(int), c->stream);
  WR_LAUNCH(wr_init_batch_info, 8, 128, c->stream, (BatchInfo*)c->batch_info, 2 * wrcu_ctx::QMAX);
  {
    const char* e = getenv("WRCU_IMMEDIATE");
    c->immediate = e && atoi(e) != 0;
    e = getenv("WRCU_PDL");
    c->pdl = e ? atoi(e) != 0 : true;
    e = getenv("WRCU_GLYPH_CTAS");
    c->glyph_ctas = e ? atoi(e) : 6;
    if (c->glyph_ctas < 1 || c->glyph_ctas > 16) c->glyph_ctas = 6;
    e = getenv("WRCU_STRIP");
    c->strip = e ? atoi(e) != 0 : true;
    e = getenv("WRCU_YUV_WIDE");
    c->yuv_wide = e && atoi(e) != 0;
    e = getenv("WRCU_EARLY_CLEAR");
    c->early_clear = e ? atoi(e) != 0 : true;
    e = getenv("WRCU_GLYPH_MAJOR");
    c->glyph_major = e ? atoi(e) != 0 : true;
    e = getenv("WRCU_SIDE_CTAS");
    c->side_ctas_per_sm = e ? atoi(e) : 1;
    if (c->side_ctas_per_sm < 1 || c->side_ctas_per_sm > 3) c->side_ctas_per_sm = 1;
    e = getenv("WRCU_STREAMS");
    c->n_streams = e ? atoi(e) : 8;
    if (c->n_streams < 1) c->n_streams = 1;
    if (c->n_streams > 32) c->n_streams = 32;
  }
#ifndef WRCU_HOSTEMU
  {  // TMA tensor maps: encoder entry point from the driver (no libcuda link), device table of records
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess && fn &&
        cudaMalloc(&c->tmaps_dev, (size_t)wrcu_ctx::TMAP_SLOTS * sizeof(CUtensorMap)) == cudaSuccess)
      c->tmap_encode = fn;
    else
      c->tmaps_dev = nullptr;
    cudaGetLastError();
  }
#endif
  {
    // shallow solid batches: up to flat_max layers go to the streaming kernel, deeper ones to the tile kernel
    // (crossover measured with tools/gpu_g.sh; WRCU_FLAT_MAX overrides it for that measurement)
    const char* e = getenv("WRCU_FLAT_MAX");
    c->flat_max = e ? atoi(e) : 2;
#ifndef WRCU_HOSTEMU
    if (c->flat_max > FLAT_MAX) c->flat_max = FLAT_MAX;
#endif
  }
  c->row_cap = 16 << 20;  // 64 MiB of row tables per batch; commands beyond it fall back to walking
  if (cudaMalloc((void**)&c->row_tab, (size_t)c->row_cap * sizeof(float)) != cudaSuccess) {
    c->row_tab = nullptr;
    c->row_cap = 0;
  }
  *out = c;
  return WRCU_OK;
}

#ifndef WRCU_HOSTEMU
static void sig_forget(const uint32_t* base, int count);
#endif
extern "C" void wrcu_ctx_destroy(wrcu_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  flush_pending(c);
  cudaStreamSynchronize(c->stream);
  for (int i = 0; i < wrcu_ctx::MAX_TEX; i++) {
    if (!c->tex[i].live) continue;
    if (!c->tex[i].imported) cudaFree(c->tex[i].dptr);
#ifndef WRCU_HOSTEMU
    else if (c->tex[i].ipc_mapped) cudaIpcCloseMemHandle(c->tex[i].dptr);
#endif
  }
#ifndef WRCU_HOSTEMU
  for (auto& pf : c->peers)
    if (pf.ipc) cudaIpcCloseMemHandle(pf.ptr);
#endif
#ifndef WRCU_HOSTEMU
  if (c->flags) sig_forget(c->flags, c->n_flags);
#endif
  if (c->flags) cudaFree(c->flags);
  for (int i = 0; i < 2; i++) {
    if (c->arena[i].host) cudaFreeHost(c->arena[i].host);
    if (c->arena[i].dev) cudaFree(c->arena[i].dev);
    if (c->arena[i].done) cudaEventDestroy(c->arena[i].done);
  }
  if (c->cmd_hot) cudaFree(c->cmd_hot);
  if (c->cmd_cold) cudaFree(c->cmd_cold);
  if (c->batch_info) cudaFree(c->batch_info);
  if (c->pool_ctr) cudaFree(c->pool_ctr);
  for (cudaStream_t st : c->side) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
  for (cudaEvent_t e : c->op_events) cudaEventDestroy(e);
  for (cudaEvent_t e : c->join_ev) cudaEventDestroy(e);
  if (c->fork_ev) cudaEventDestroy(c->fork_ev);
  if (c->fork0_ev) cudaEventDestroy(c->fork0_ev);
  delete (std::vector<PendingOp>*)c->pending_ops;
  if (c->row_tab) cudaFree(c->row_tab);
  if (c->tmaps_dev) cudaFree(c->tmaps_dev);
  if (c->fail_pool) cudaFree(c->fail_pool);
  if (c->gpu_cache_dev) cudaFree(c->gpu_cache_dev);
  if (c->dev_err) cudaFree(c->dev_err);
  if (c->bin_mask) cudaFree(c->bin_mask);
  if (c->t0) cudaEventDestroy(c->t0);
  if (c->t1) cudaEventDestroy(c->t1);
  if (c->p0) cudaEventDestroy(c->p0);
  if (c->p1) cudaEventDestroy(c->p1);
  if (c->copy_stream) {
    cudaStreamSynchronize(c->copy_stream);
    cudaStreamDestroy(c->copy_stream);
    cudaEventDestroy(c->ready_ev);
    for (int i = 0; i < wrcu_ctx::N_FENCES; i++) cudaEventDestroy(c->fence_ev[i]);
  }
  cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" int wrcu_get_error(wrcu_ctx* c) {
  int e = c->sticky_error;
  c->sticky_error = 0;
  return e;
}
extern "C" const char* wrcu_last_error_string(wrcu_ctx* c) { return c ? c->err : "no context"; }

static int sync_and_check(wrcu_ctx* c);
extern "C" int wrcu_finish(wrcu_ctx* c) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  cudaSetDevice(c->device);
  int rc = sync_and_check(c);
  if (c->copy_stream) WRCU_CUDA(c, cudaStreamSynchronize(c->copy_stream));
  return rc;
}

extern "C" int wrcu_stream(wrcu_ctx* c, void** stream) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  *stream = (void*)c->stream;
  return WRCU_OK;
}

// ---- arena ---------------------------------------------------------------------------
// Stage `bytes` of host data for the device: copy into the pinned arena (so the
// caller may free its buffer on return) and queue the H2D copy on the stream.
// Reserve `bytes` in the current arena (host and device side at the same offset).
static int flush_pending(wrcu_ctx* c);
static void mark_dirty(wrcu_ctx* c, size_t lo, size_t hi) {
  if (c->dirty_hi <= c->dirty_lo) { c->dirty_lo = lo; c->dirty_hi = hi; return; }
  if (lo < c->dirty_lo) c->dirty_lo = lo;
  if (hi > c->dirty_hi) c->dirty_hi = hi;
}
static int arena_reserve(wrcu_ctx* c, size_t bytes, size_t* off_out) {
  Arena* a = &c->arena[c->cur_arena];
  size_t off = align_up(a->used, 256);
  if (off + bytes > a->cap) {
    // queued batches hold pointers into this arena: run them before it moves
    { int rcf = flush_pending(c); if (rcf != WRCU_OK) return rcf; }
    a = &c->arena[c->cur_arena];
    off = align_up(a->used, 256);
    // grow: finish outstanding work, then reallocate this arena larger
    WRCU_CUDA(c, cudaStreamSynchronize(c->stream));
    size_t ncap = align_up((off + bytes) * 2, 1u << 20);
    uint8_t *nh = nullptr, *nd = nullptr;
    WRCU_CUDA(c, cudaMallocHost((void**)&nh, ncap));
    WRCU_CUDA(c, cudaMalloc((void**)&nd, ncap));
    // earlier stagings of this frame are still referenced by queued kernels →
    // they have completed (we synchronised), but tables may be used by later
    // draws: keep contents by copying.
    memcpy(nh, a->host, a->used);
    WRCU_CUDA(c, cudaMemcpy(nd, a->dev, a->used, cudaMemcpyDeviceToDevice));
    // rebase table pointers
    ptrdiff_t delta = nd - a->dev;
#define REBASE(p) if (p) p = (decltype(p))((uint8_t*)(p) + delta)
    REBASE(c->tables.prim_headers_f); REBASE(c->tables.prim_headers_i);
    REBASE(c->tables.transforms); REBASE(c->tables.render_tasks);
    if (!c->gpu_cache_bound) REBASE(c->tables.gpu_cache);
    REBASE(c->tables.gpu_buffer_f); REBASE(c->tables.gpu_buffer_i);
#undef REBASE
    cudaFreeHost(a->host);
    cudaFree(a->dev);
    a->host = nh;
    a->dev = nd;
    a->cap = ncap;
  }
  a->used = off + bytes;
  *off_out = off;
  return WRCU_OK;
}

// `zero_copy_ok`: only the texture-upload entry points pass true — their header contract says a
// wrcu_host_alloc buffer stays busy until a fence taken after the call (wrcu_fence_insert) has been
// waited on.  Instances, tables and texture lists are ALWAYS copied into the arena before the call
// returns (glBufferData ownership, include/wrcu.h conventions).
// `defer`: the data is only read by kernels launched from flush_pending — no copy of its own, the arena range
// [dirty_lo, dirty_hi) goes to the device in ONE cudaMemcpyAsync there (a page's 150 instance arrays and its
// tables travel together instead of as 150 copy-engine operations).
static int stage(wrcu_ctx* c, const void* src, size_t bytes, void** dev_out, bool zero_copy_ok = false, bool defer = false) {
  size_t off = 0;
  int rc = arena_reserve(c, bytes, &off);
  if (rc != WRCU_OK) return rc;
  Arena* a = &c->arena[c->cur_arena];
  // page-locked memory handed out by wrcu_host_alloc goes to the device directly (the mapped-PBO
  // case of the reference's upload path); anything else is first copied into the pinned arena
  bool pinned = false;
  if (zero_copy_ok)
  for (const auto& ha : c->host_allocs)
    if ((const uint8_t*)src >= ha.first && (const uint8_t*)src + bytes <= ha.first + ha.second) { pinned = true; break; }
  if (pinned) {
    WRCU_CUDA(c, cudaMemcpyAsync(a->dev + off, src, bytes, cudaMemcpyHostToDevice, c->stream));
  } else {
    memcpy(a->host + off, src, bytes);
    if (defer) mark_dirty(c, off, off + bytes);
    else WRCU_CUDA(c, cudaMemcpyAsync(a->dev + off, a->host + off, bytes, cudaMemcpyHostToDevice, c->stream));
  }
  c->stats.h2d_bytes += bytes;
  *dev_out = a->dev + off;
  return WRCU_OK;
}

// ---- textures ----------------------------------------------------------------------
static void make_tensor_map(wrcu_ctx* c, int id);
extern "C" int wrcu_texture_create(wrcu_ctx* c, int format, int w, int h, wrcu_tex* out) {
  int bpp = fmt_bpp(format);
  if (!bpp || w <= 0 || h <= 0 || w > 32767 || h > 32767 || !out)
    return wrcu_fail(c, WRCU_ERR_INVALID, "texture_create: bad arguments");
  cudaSetDevice(c->device);
  for (int i = 1; i < wrcu_ctx::MAX_TEX; i++) {
    if (!c->tex[i].live) {
      WrTexture& t = c->tex[i];
      t.fmt = format; t.w = w; t.h = h; t.bpp = bpp; t.filter = WRCU_LINEAR;
      // pitch covers whole raster tiles so tile-wide vector accesses stay inside
      // the allocation; rows padded to tile height likewise.
      t.pitch = align_up((size_t)align_up(w, WRCU_TILE_W) * bpp, 256);
      size_t rows = align_up(h, WRCU_TILE_H);
      WRCU_CUDA(c, cudaMalloc((void**)&t.dptr, t.pitch * rows));
      WRCU_CUDA(c, cudaMemsetAsync(t.dptr, 0, t.pitch * rows, c->stream));
      t.live = true;
      make_tensor_map(c, i);
      *out = (wrcu_tex)i;
      return WRCU_OK;
    }
  }
  return wrcu_fail(c, WRCU_ERR_OOM, "texture_create: out of texture handles");
}

#ifndef WRCU_HOSTEMU
// One 2-D tensor map per RGBA8 texture: u32 elements, box WR_TMA_BOX_W x WR_TMA_BOX_H, no swizzle
// (the boxes are only ever moved, never read by threads).  The 128-byte record is built on the host
// and copied into the next FRESH slot of the context's device table (TexView::tmap_id = the slot);
// kernels address it as tmaps + slot.  A slot is never rewritten until the table wraps (65535 texture
// creations), so no SM can hold a stale copy of a descriptor and the copy kernels need no
// tensormap-proxy acquire — one per source texture and CTA had made that kernel's start-up its whole
// cost.  After a wrap the kernels are told to acquire (RasterArgs::tmap_acquire).
static void make_tensor_map(wrcu_ctx* c, int id) {
  WrTexture& t = c->tex[id];
  t.has_tmap = false;
  t.tmap_slot = 0;
  if (!c->tmap_encode || !c->tmaps_dev || t.fmt != WRCU_FMT_RGBA8 || t.w < WR_TMA_BOX_W || t.h < WR_TMA_BOX_H) return;
  CUtensorMap m;
  const cuuint64_t dims[2] = {(cuuint64_t)t.w, (cuuint64_t)t.h};
  const cuuint64_t strides[1] = {(cuuint64_t)t.pitch};
  const cuuint32_t box[2] = {WR_TMA_BOX_W, WR_TMA_BOX_H};
  const cuuint32_t estr[2] = {1, 1};
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  CUresult r = ((EncodeFn)c->tmap_encode)(&m, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, t.dptr, dims, strides, box, estr,
                                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return;
  int slot = c->tmap_next++;
  if (slot >= wrcu_ctx::TMAP_SLOTS) {
    c->tmap_wrapped = true;
    slot = 1;
    c->tmap_next = 2;
  }
  if (cudaMemcpyAsync((uint8_t*)c->tmaps_dev + (size_t)slot * sizeof(CUtensorMap), &m, sizeof m, cudaMemcpyHostToDevice,
                      c->stream) != cudaSuccess)
    return;
  t.tmap_slot = slot;
  t.has_tmap = true;
}
#else
// host emulation: no copy engine, but the copy-class decision of the setup stage still runs (tests)
static void make_tensor_map(wrcu_ctx* c, int id) {
  WrTexture& t = c->tex[id];
  t.has_tmap = t.fmt == WRCU_FMT_RGBA8 && t.w >= 256 && t.h >= 16;
  t.tmap_slot = t.has_tmap ? id : 0;
}
#endif

static WrTexture* get_tex(wrcu_ctx* c, wrcu_tex id) {
  return (id > 0 && id < wrcu_ctx::MAX_TEX && c->tex[id].live) ? &c->tex[id] : nullptr;
}

extern "C" int wrcu_texture_set_filter(wrcu_ctx* c, wrcu_tex id, int filter) {
  WrTexture* t = get_tex(c, id);
  if (!t) return wrcu_fail(c, WRCU_ERR_INVALID, "texture_set_filter: bad handle");
  t->filter = filter;
  return WRCU_OK;
}

extern "C" int wrcu_texture_upload(wrcu_ctx* c, wrcu_tex id, int x, int y, int w, int h,
                                   const void* data, size_t src_stride) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture* t = get_tex(c, id);
  if (!t || !data || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > t->w || y + h > t->h)
    return wrcu_fail(c, WRCU_ERR_INVALID, "texture_upload: bad arguments");
  cudaSetDevice(c->device);
  size_t row = (size_t)w * t->bpp;
  // pack rows tightly into the pinned arena, then one strided async copy
  Arena* a = &c->arena[c->cur_arena];
  size_t need = row * h;
  void* dsrc = nullptr;
  if (src_stride == row) {
    int rc = stage(c, data, need, &dsrc, true);
    if (rc) return rc;
  } else {
    // stage row by row (host memcpy), single device copy
    uint8_t* tmp = (uint8_t*)malloc(need);
    if (!tmp) return wrcu_fail(c, WRCU_ERR_OOM, "texture_upload: host oom");
    for (int r = 0; r < h; r++) memcpy(tmp + r * row, (const uint8_t*)data + (size_t)r * src_stride, row);
    int rc = stage(c, tmp, need, &dsrc);
    free(tmp);
    if (rc) return rc;
  }
  (void)a;
  WRCU_CUDA(c, cudaMemcpy2DAsync(t->dptr + (size_t)y * t->pitch + (size_t)x * t->bpp, t->pitch, dsrc, row,
                                 row, h, cudaMemcpyDeviceToDevice, c->stream));
  return WRCU_OK;
}

extern "C" int wrcu_texture_destroy(wrcu_ctx* c, wrcu_tex id) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture* t = get_tex(c, id);
  if (!t) return wrcu_fail(c, WRCU_ERR_INVALID, "texture_destroy: bad handle");
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (!t->imported) cudaFree(t->dptr);
#ifndef WRCU_HOSTEMU
  else if (t->ipc_mapped) cudaIpcCloseMemHandle(t->dptr);
#endif
  *t = WrTexture();
  if (c->color_tex == id) c->color_tex = 0;
  if (c->depth_tex == id) c->depth_tex = 0;
  return WRCU_OK;
}

extern "C" int wrcu_texture_device_ptr(wrcu_ctx* c, wrcu_tex id, void** dptr, size_t* pitch) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture* t = get_tex(c, id);
  if (!t) return wrcu_fail(c, WRCU_ERR_INVALID, "texture_device_ptr: bad handle");
  *dptr = t->dptr;
  *pitch = t->pitch;
  return WRCU_OK;
}

// Synchronise and surface instances the setup kernels could not rasterise
// (rotated / perspective quads): reported once, as WRCU_ERR_UNSUPPORTED.
static int sync_and_check(wrcu_ctx* c) {
  int n = 0;
  WRCU_CUDA(c, cudaMemcpyAsync(&n, c->dev_err, sizeof n, cudaMemcpyDeviceToHost, c->stream));
  WRCU_CUDA(c, cudaStreamSynchronize(c->stream));
  if (n >= (1 << 20)) {
    cudaMemsetAsync(c->dev_err, 0, sizeof(int), c->stream);
    return wrcu_fail(c, WRCU_ERR_CUDA, "wrcu_peer_wait: a peer did not signal within 2 s (%d wait(s) timed out; counter 0x%x, "
                     "%d polling waits and %d event waits queued by this context)", n >> 20, n, c->n_wait_kernel, c->n_wait_event);
  }
  if (n) {
    cudaMemsetAsync(c->dev_err, 0, sizeof(int), c->stream);
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED,
                     "%d instance(s) not rasterised: perspective under a kind without the per-sample 1/w path, or resources exhausted", n);
  }
  return WRCU_OK;
}

extern "C" int wrcu_read_pixels(wrcu_ctx* c, wrcu_tex id, int x, int y, int w, int h, void* out,
                                size_t dst_stride) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture* t = get_tex(c, id);
  if (!t || !out || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > t->w || y + h > t->h)
    return wrcu_fail(c, WRCU_ERR_INVALID, "read_pixels: bad arguments");
  cudaSetDevice(c->device);
  size_t row = (size_t)w * t->bpp;
  WRCU_CUDA(c, cudaMemcpy2DAsync(out, dst_stride, t->dptr + (size_t)y * t->pitch + (size_t)x * t->bpp,
                                 t->pitch, row, h, cudaMemcpyDeviceToHost, c->stream));
  c->stats.d2h_bytes += row * h;
  return sync_and_check(c);
}

// ---- asynchronous readback ---------------------------------------------------------------
extern "C" int wrcu_host_alloc(wrcu_ctx* c, size_t bytes, void** out) {
  if (!out || bytes == 0) return wrcu_fail(c, WRCU_ERR_INVALID, "host_alloc: bad arguments");
  cudaSetDevice(c->device);
  WRCU_CUDA(c, cudaMallocHost(out, bytes));
  c->host_allocs.push_back(std::make_pair((uint8_t*)*out, bytes));
  return WRCU_OK;
}
extern "C" int wrcu_host_free(wrcu_ctx* c, void* ptr) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  if (!ptr) return WRCU_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);  // a staged copy may still be reading it
  for (size_t i = 0; i < c->host_allocs.size(); i++)
    if (c->host_allocs[i].first == (uint8_t*)ptr) { c->host_allocs.erase(c->host_allocs.begin() + i); break; }
  cudaFreeHost(ptr);
  return WRCU_OK;
}

static int ensure_copy_stream(wrcu_ctx* c);
static int wait_fence(wrcu_ctx* c, uint64_t fence, bool on_stream) {
  if (fence == 0) return WRCU_OK;
  int slot = (int)(fence % wrcu_ctx::N_FENCES);
  if (c->fence_id[slot] != fence) return WRCU_OK;  // slot recycled: that copy completed long ago
  if (on_stream) WRCU_CUDA(c, cudaStreamWaitEvent(c->stream, c->fence_ev[slot], 0));
  else WRCU_CUDA(c, cudaEventSynchronize(c->fence_ev[slot]));
  return WRCU_OK;
}

extern "C" int wrcu_read_pixels_async(wrcu_ctx* c, wrcu_tex id, int x, int y, int w, int h, void* out,
                                      size_t dst_stride, uint64_t* fence) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture* t = get_tex(c, id);
  if (!t || !out || !fence || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > t->w || y + h > t->h)
    return wrcu_fail(c, WRCU_ERR_INVALID, "read_pixels_async: bad arguments");
  cudaSetDevice(c->device);
  { int rce = ensure_copy_stream(c); if (rce != WRCU_OK) return rce; }
  uint64_t id64 = c->next_fence++;
  int slot = (int)(id64 % wrcu_ctx::N_FENCES);
  if (c->fence_id[slot]) WRCU_CUDA(c, cudaEventSynchronize(c->fence_ev[slot]));  // ring wrapped: oldest copy must be done
  size_t row = (size_t)w * t->bpp;
  WRCU_CUDA(c, cudaEventRecord(c->ready_ev, c->stream));
  WRCU_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ready_ev, 0));
  WRCU_CUDA(c, cudaMemcpy2DAsync(out, dst_stride, t->dptr + (size_t)y * t->pitch + (size_t)x * t->bpp, t->pitch, row, h,
                                 cudaMemcpyDeviceToHost, c->copy_stream));
  WRCU_CUDA(c, cudaEventRecord(c->fence_ev[slot], c->copy_stream));
  c->fence_id[slot] = id64;
  t->pending_read = id64;
  c->stats.d2h_bytes += row * h;
  *fence = id64;
  return WRCU_OK;
}

static int ensure_copy_stream(wrcu_ctx* c) {
  if (c->copy_stream) return WRCU_OK;
  WRCU_CUDA(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  WRCU_CUDA(c, cudaEventCreateWithFlags(&c->ready_ev, cudaEventDisableTiming));
  for (int i = 0; i < wrcu_ctx::N_FENCES; i++)
    WRCU_CUDA(c, cudaEventCreateWithFlags(&c->fence_ev[i], cudaEventDisableTiming));
  return WRCU_OK;
}

// glFenceSync on the draw stream: everything queued so far (uploads reading wrcu_host_alloc memory
// included) has completed once wrcu_fence_wait(fence) returns.
extern "C" int wrcu_fence_insert(wrcu_ctx* c, uint64_t* fence) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  if (!fence) return wrcu_fail(c, WRCU_ERR_INVALID, "fence_insert: null fence");
  cudaSetDevice(c->device);
  int rc = ensure_copy_stream(c);
  if (rc != WRCU_OK) return rc;
  uint64_t id64 = c->next_fence++;
  int slot = (int)(id64 % wrcu_ctx::N_FENCES);
  if (c->fence_id[slot]) WRCU_CUDA(c, cudaEventSynchronize(c->fence_ev[slot]));
  WRCU_CUDA(c, cudaEventRecord(c->fence_ev[slot], c->stream));
  c->fence_id[slot] = id64;
  *fence = id64;
  return WRCU_OK;
}

extern "C" int wrcu_fence_wait(wrcu_ctx* c, uint64_t fence) {
  cudaSetDevice(c->device);
  int rc = wait_fence(c, fence, false);
  if (rc != WRCU_OK) return rc;
  return WRCU_OK;
}

// ---- update path ---------------------------------------------------------------------
extern "C" int wrcu_texture_upload_batch(wrcu_ctx* c, wrcu_tex id, const wrcu_upload_rect* rects, size_t n,
                                         const void* staging, size_t staging_bytes) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture* t = get_tex(c, id);
  if (!t || (n && (!rects || !staging))) return wrcu_fail(c, WRCU_ERR_INVALID, "texture_upload_batch: bad arguments");
  if (!n) return WRCU_OK;
  for (size_t i = 0; i < n; i++) {
    const wrcu_upload_rect& r = rects[i];
    size_t row = (size_t)r.w * t->bpp;
    if (r.x < 0 || r.y < 0 || r.w <= 0 || r.h <= 0 || r.x + r.w > t->w || r.y + r.h > t->h || r.stride < row ||
        r.offset + (size_t)(r.h - 1) * r.stride + row > staging_bytes)
      return wrcu_fail(c, WRCU_ERR_INVALID, "texture_upload_batch: rect %zu out of range", i);
  }
  cudaSetDevice(c->device);
  if (t->pending_read) {
    int rc0 = wait_fence(c, t->pending_read, true);
    if (rc0 != WRCU_OK) return rc0;
    t->pending_read = 0;
  }
  int rc;
  void *dstage = nullptr, *drects = nullptr;
  if ((rc = stage(c, staging, staging_bytes, &dstage, true)) != WRCU_OK) return rc;
  std::vector<UploadRectDev> hr(n);
  int max_h = 1;
  for (size_t i = 0; i < n; i++) {
    hr[i] = UploadRectDev{rects[i].x, rects[i].y, rects[i].w, rects[i].h, rects[i].offset, rects[i].stride};
    max_h = max(max_h, rects[i].h);
  }
  // the second stage() may grow (reallocate) the arena: keep the blob by offset
  Arena* a = &c->arena[c->cur_arena];
  const size_t blob_off = (size_t)((uint8_t*)dstage - a->dev);
  if ((rc = stage(c, hr.data(), n * sizeof(UploadRectDev), &drects)) != WRCU_OK) return rc;
  dstage = a->dev + blob_off;
  dim3 grid((unsigned)n, (unsigned)min(max_h, 64));
  WR_LAUNCH(wr_upload_scatter, grid, 128, c->stream, t->dptr, (int)t->pitch, t->bpp, (const UploadRectDev*)drects,
            (int)n, (const uint8_t*)dstage);
  c->stats.kernel_launches++;
  WRCU_CUDA(c, cudaGetLastError());
  return WRCU_OK;
}

extern "C" int wrcu_texture_copy(wrcu_ctx* c, wrcu_tex src, wrcu_tex dst, const int32_t r[4], int dx, int dy) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture *s = get_tex(c, src), *d = get_tex(c, dst);
  if (!s || !d || !r || s->bpp != d->bpp || r[2] <= 0 || r[3] <= 0 || r[0] < 0 || r[1] < 0 || r[0] + r[2] > s->w ||
      r[1] + r[3] > s->h || dx < 0 || dy < 0 || dx + r[2] > d->w || dy + r[3] > d->h)
    return wrcu_fail(c, WRCU_ERR_INVALID, "texture_copy: bad arguments");
  cudaSetDevice(c->device);
  WRCU_CUDA(c, cudaMemcpy2DAsync(d->dptr + (size_t)dy * d->pitch + (size_t)dx * d->bpp, d->pitch,
                                 s->dptr + (size_t)r[1] * s->pitch + (size_t)r[0] * s->bpp, s->pitch,
                                 (size_t)r[2] * s->bpp, r[3], cudaMemcpyDeviceToDevice, c->stream));
  return WRCU_OK;
}

extern "C" int wrcu_gpu_cache_update(wrcu_ctx* c, int height, int clear, const wrcu_gpu_cache_copy* updates,
                                     size_t n_updates, const float* blocks, size_t n_blocks) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  if (height <= 0 || height > 65536 || (n_updates && (!updates || !blocks)))
    return wrcu_fail(c, WRCU_ERR_INVALID, "gpu_cache_update: bad arguments");
  cudaSetDevice(c->device);
  if (height > c->gpu_cache_rows) {  // ensure_texture (renderer/gpu_cache.rs:103-155): grow, keep contents
    float4* n = nullptr;
    WRCU_CUDA(c, cudaMalloc((void**)&n, (size_t)height * 1024 * sizeof(float4)));
    WRCU_CUDA(c, cudaMemsetAsync(n, 0, (size_t)height * 1024 * sizeof(float4), c->stream));
    if (c->gpu_cache_dev) {
      WRCU_CUDA(c, cudaMemcpyAsync(n, c->gpu_cache_dev, (size_t)c->gpu_cache_rows * 1024 * sizeof(float4),
                                   cudaMemcpyDeviceToDevice, c->stream));
      WRCU_CUDA(c, cudaStreamSynchronize(c->stream));
      cudaFree(c->gpu_cache_dev);
    }
    if (c->gpu_cache_bound) c->tables.gpu_cache = n;
    c->gpu_cache_dev = n;
    c->gpu_cache_rows = height;
    if (c->gpu_cache_bound) c->tables.n_gpu_cache = height * 1024;
  }
  if (clear)
    WRCU_CUDA(c, cudaMemsetAsync(c->gpu_cache_dev, 0, (size_t)c->gpu_cache_rows * 1024 * sizeof(float4), c->stream));
  if (!n_updates) return WRCU_OK;
  for (size_t i = 0; i < n_updates; i++)
    if ((size_t)updates[i].block_index + updates[i].block_count > n_blocks || updates[i].v >= c->gpu_cache_rows ||
        updates[i].u + updates[i].block_count > 1024)
      return wrcu_fail(c, WRCU_ERR_INVALID, "gpu_cache_update: update %zu out of range", i);
  int rc;
  void *dblocks = nullptr, *dupd = nullptr;
  if ((rc = stage(c, blocks, n_blocks * 16, &dblocks)) != WRCU_OK) return rc;
  static_assert(sizeof(wrcu_gpu_cache_copy) == sizeof(GpuCacheCopyDev), "update record layout");
  Arena* a = &c->arena[c->cur_arena];
  const size_t blocks_off = (size_t)((uint8_t*)dblocks - a->dev);
  if ((rc = stage(c, updates, n_updates * sizeof(wrcu_gpu_cache_copy), &dupd)) != WRCU_OK) return rc;
  dblocks = a->dev + blocks_off;
  int threads = 128, warps_per_block = threads / 32;
  int grid = (int)((n_updates + warps_per_block - 1) / warps_per_block);
  WR_LAUNCH(wr_gpu_cache_scatter, grid, threads, c->stream, c->gpu_cache_dev, c->gpu_cache_rows,
            (const GpuCacheCopyDev*)dupd, (int)n_updates, (const float4*)dblocks, (int)n_blocks);
  c->stats.kernel_launches++;
  WRCU_CUDA(c, cudaGetLastError());
  return WRCU_OK;
}

// ---- SwCompositor blit (swgl/src/composite.h:166-417, 532-590) -----------------------------------
static int wait_pending_read(wrcu_ctx* c, WrTexture* t);
static TexView tex_view(wrcu_ctx* c, wrcu_tex id);
struct BlitArgs {
  uint8_t* dst; int dst_pitch;
  TexView src;
  int dx0, dy0;                 // dstReq origin
  int bx0, by0, bx1, by1;       // dstBounds, relative to dstReq
  int sx0, sy0, sy1;            // srcReq.x0, .y0, .y1
  // nearest: first source column/row (relative to srcReq) and the Bresenham fractions at dstBounds' corner
  int sbx0, sby0, fracx0, fracy0, sw, sh, dw, dh, invert_y;
  // linear: quantised uv at dstBounds' corner and per-pixel / per-row steps (x128)
  float u0, v0, du, dv;
  int opaque, linear;
};
WRD uint32_t wr_blit_over(uint32_t d, uint32_t s) {  // srcpx + dstpx - muldiv255(dstpx, alphas(srcpx)), saturating pack
  const uint32_t cc = 255u - (s >> 24);
  const uint32_t rb = wr_premult_over_pair(d & 0x00FF00FFu, s & 0x00FF00FFu, cc);
  const uint32_t ga = wr_premult_over_pair((d >> 8) & 0x00FF00FFu, (s >> 8) & 0x00FF00FFu, cc);
  return rb | (ga << 8);
}
WRD void wr_blit_pixel(const BlitArgs& a, int x, int y) {  // x, y relative to dstReq, inside dstBounds
  uint32_t s;
  if (!a.linear) {
    // scale_row / the row stepping of scale_blit in closed form: `for (frac += srcW; frac >= dstW; frac -= dstW) src++`
    const int col = a.sbx0 + (a.fracx0 + a.sw * (x - a.bx0)) / a.dw;
    const int row = a.sby0 + (a.fracy0 + a.sh * (y - a.by0)) / a.dh;
    const int sy = a.invert_y ? a.sy1 - 1 - row : a.sy0 + row;
    s = *(const uint32_t*)(a.src.ptr + (size_t)sy * a.src.pitch + (size_t)(a.sx0 + col) * 4);
  } else {
    // linear_row_blit: uv = init_interp(srcUV, (srcDU, 0)); per 4-pixel chunk uv.x += 4 * srcDU; rows srcUV.y += srcDUV.y
    const int i = x - a.bx0, j = i & 3, k = i >> 2;
    float u = a.u0;
    for (int q = 0; q < j; q++) u = __fadd_rn(u, a.du);
    u = wr_repeat_add(u, __fmul_rn(4.0f, a.du), k);
    const float v = wr_repeat_add(a.v0, a.dv, y - a.by0);
    const Px p = wr_texture_linear_rgba8(a.src, (int)u, (int)v);
    s = (uint32_t)wr_pack16(p.b) | ((uint32_t)wr_pack16(p.g) << 8) | ((uint32_t)wr_pack16(p.r) << 16) | ((uint32_t)wr_pack16(p.a) << 24);
  }
  uint32_t* d = (uint32_t*)(a.dst + (size_t)(a.dy0 + y) * a.dst_pitch) + a.dx0 + x;
  *d = a.opaque ? s : wr_blit_over(*d, s);
}
#ifdef WRCU_HOSTEMU
static void wr_sw_composite_blit(BlitArgs a) {
  for (int y = a.by0; y < a.by1; y++)
    for (int x = a.bx0; x < a.bx1; x++) wr_blit_pixel(a, x, y);
}
#else
__global__ void wr_sw_composite_blit(BlitArgs a) {
  const int x = a.bx0 + blockIdx.x * blockDim.x + threadIdx.x, y = a.by0 + blockIdx.y * blockDim.y + threadIdx.y;
  if (x < a.bx1 && y < a.by1) wr_blit_pixel(a, x, y);
}
#endif

struct IRect { int x0, y0, x1, y1; };
static IRect irect_intersect(IRect a, IRect b) {
  return IRect{a.x0 > b.x0 ? a.x0 : b.x0, a.y0 > b.y0 ? a.y0 : b.y0, a.x1 < b.x1 ? a.x1 : b.x1, a.y1 < b.y1 ? a.y1 : b.y1};
}
extern "C" int wrcu_composite_blit(wrcu_ctx* c, wrcu_tex dst_id, wrcu_tex src_id, const int32_t sr[4], const int32_t dr[4],
                                   int opaque, int flip_x, int flip_y, int filter_linear, const int32_t cr[4]) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture *d = get_tex(c, dst_id), *s = get_tex(c, src_id);
  if (!d || !s || !sr || !dr || !cr || d->fmt != WRCU_FMT_RGBA8 || s->fmt != WRCU_FMT_RGBA8)
    return wrcu_fail(c, WRCU_ERR_INVALID, "composite_blit: needs two RGBA8 textures and three rects");
  cudaSetDevice(c->device);
  { int rcw = wait_pending_read(c, d); if (rcw != WRCU_OK) return rcw; }
  const IRect srcReq{sr[0], sr[1], sr[0] + sr[2], sr[1] + sr[3]}, dstReq{dr[0], dr[1], dr[0] + dr[2], dr[1] + dr[3]};
  if (srcReq.x1 <= srcReq.x0 || srcReq.y1 <= srcReq.y0 || dstReq.x1 <= dstReq.x0 || dstReq.y1 <= dstReq.y0) return WRCU_OK;
  const IRect clip{cr[0] - dr[0], cr[1] - dr[1], cr[0] - dr[0] + cr[2], cr[1] - dr[1] + cr[3]};  // relative to dstReq
  const int sw = sr[2], sh = sr[3], dw = dr[2], dh = dr[3];
  const bool same = sw == dw && sh == dh;
  const bool linear = s->w >= 2 && (flip_x || (!same && filter_linear));
  BlitArgs a;
  memset(&a, 0, sizeof a);
  a.dst = d->dptr; a.dst_pitch = (int)d->pitch;
  a.src = tex_view(c, src_id);
  a.src.filter = WRCU_LINEAR;
  a.dx0 = dstReq.x0; a.dy0 = dstReq.y0;
  a.sx0 = srcReq.x0; a.sy0 = srcReq.y0; a.sy1 = srcReq.y1;
  a.sw = sw; a.sh = sh; a.dw = dw; a.dh = dh;
  a.opaque = opaque ? 1 : 0;
  a.linear = linear ? 1 : 0;
  a.invert_y = flip_y ? 1 : 0;
  // dsttex.sample_bounds(dstReq) ∩ clipRect (Texture::sample_bounds, gl.cc:554-558)
  IRect db = irect_intersect(IRect{0, 0, d->w, d->h}, dstReq);
  db = IRect{db.x0 - dstReq.x0, db.y0 - dstReq.y0, db.x1 - dstReq.x0, db.y1 - dstReq.y0};
  db = irect_intersect(db, clip);
  if (linear) {
    if (db.x1 <= db.x0 || db.y1 <= db.y0) return WRCU_OK;
    float su = (float)srcReq.x0, sv = (float)srcReq.y0;
    float du = (float)sw / (float)dw, dv = (float)sh / (float)dh;
    if (flip_x) { su += (float)sw; du = -du; }
    if (flip_y) { sv += (float)sh; dv = -dv; }
    su += du * ((float)db.x0 + 0.5f);
    sv += dv * ((float)db.y0 + 0.5f);
    a.u0 = su * 128.0f + (0.5f - 0.5f * 128.0f);  // linearQuantize(srcUV, 128) (texture.h:428-430)
    a.v0 = sv * 128.0f + (0.5f - 0.5f * 128.0f);
    a.du = du * 128.0f;
    a.dv = dv * 128.0f;
  } else {
    // scale_blit (composite.h:166-282): limit the destination so that no sample falls outside the source
    IRect sb = irect_intersect(IRect{0, 0, s->w, s->h}, srcReq);
    sb = IRect{sb.x0 - srcReq.x0, sb.y0 - srcReq.y0, sb.x1 - srcReq.x0, sb.y1 - srcReq.y0};
    if (flip_y) { const int t0 = sh - sb.y1, t1 = sh - sb.y0; sb.y0 = t0; sb.y1 = t1; }  // invert_y
    IRect sc{0 - srcReq.x0, 0 - srcReq.y0, s->w - srcReq.x0, s->h - srcReq.y0};  // srctex.bounds() - srcReq.origin()
    if (flip_y) { const int t0 = sh - sc.y1, t1 = sh - sc.y0; sc.y0 = t0; sc.y1 = t1; }
    // IntRect::scale(srcW, srcH, dstW, dstH, roundIn = true) (gl.cc:143-150), C integer division as there
    sc = IRect{(sc.x0 * dw + (sw - 1)) / sw, (sc.y0 * dh + (sh - 1)) / sh, (sc.x1 * dw) / sw, (sc.y1 * dh) / sh};
    db = irect_intersect(db, sc);
    if (db.x1 <= db.x0 || db.y1 <= db.y0) return WRCU_OK;
    const int fx = sw * db.x0, fy = sh * db.y0;
    a.sbx0 = fx / dw > sb.x0 ? fx / dw : sb.x0;
    a.sby0 = fy / dh > sb.y0 ? fy / dh : sb.y0;
    a.fracx0 = fx % dw;
    a.fracy0 = fy % dh;
  }
  a.bx0 = db.x0; a.by0 = db.y0; a.bx1 = db.x1; a.by1 = db.y1;
#ifdef WRCU_HOSTEMU
  wr_sw_composite_blit(a);
#else
  dim3 block(64, 4), grid((unsigned)((db.x1 - db.x0 + 63) / 64), (unsigned)((db.y1 - db.y0 + 3) / 4));
  wr_sw_composite_blit<<<grid, block, 0, c->stream>>>(a);
  WRCU_CUDA(c, cudaGetLastError());
#endif
  c->stats.kernel_launches++;
  return WRCU_OK;
}

// ---- SwCompositor YUV blit (swgl/src/composite.h:1146-1205, 1335-1384) --------------------------
extern "C" int wrcu_composite_blit_yuv(wrcu_ctx* c, wrcu_tex dst_id, wrcu_tex y_id, wrcu_tex u_id, wrcu_tex v_id,
                                       int color_space, uint32_t color_depth, const int32_t sr[4], const int32_t dr[4],
                                       int flip_x, int flip_y, const int32_t cr[4]) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WrTexture *d = get_tex(c, dst_id), *ty = get_tex(c, y_id), *tu = get_tex(c, u_id), *tv = get_tex(c, v_id);
  if (!d || !ty || !tu || !tv || !sr || !dr || !cr || d->fmt != WRCU_FMT_RGBA8 || color_space < 0 || color_space > 6)
    return wrcu_fail(c, WRCU_ERR_INVALID, "composite_blit_yuv: needs an RGBA8 destination, three planes, three rects, a colour space 0..6");
  const bool r8 = ty->fmt == WRCU_FMT_R8 && tu->fmt == WRCU_FMT_R8 && tv->fmt == WRCU_FMT_R8 && color_depth == 8;
  const bool r16 = ty->fmt == WRCU_FMT_R16 && tu->fmt == WRCU_FMT_R16 && tv->fmt == WRCU_FMT_R16 &&
                   (color_depth == 10 || color_depth == 12 || color_depth == 16);
  if (!r8 && !r16)
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "composite_blit_yuv: three R8 planes at depth 8, or three R16 planes at depth 10, 12 or 16");
  if (tu->w != tv->w || tu->h != tv->h || tu->pitch != tv->pitch)
    return wrcu_fail(c, WRCU_ERR_INVALID, "composite_blit_yuv: the chroma planes must have one size");
  if (ty->w < 2 || tu->w < 2)
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "composite_blit_yuv: planes under 2 texels wide (the reference's single-texel fill)");
  cudaSetDevice(c->device);
  { int rcw = wait_pending_read(c, d); if (rcw != WRCU_OK) return rcw; }
  const IRect srcReq{sr[0], sr[1], sr[0] + sr[2], sr[1] + sr[3]}, dstReq{dr[0], dr[1], dr[0] + dr[2], dr[1] + dr[3]};
  if (srcReq.x1 <= srcReq.x0 || srcReq.y1 <= srcReq.y0 || dstReq.x1 <= dstReq.x0 || dstReq.y1 <= dstReq.y0) return WRCU_OK;
  const IRect clip{cr[0] - dr[0], cr[1] - dr[1], cr[0] - dr[0] + cr[2], cr[1] - dr[1] + cr[3]};  // relative to dstReq
  IRect db = irect_intersect(IRect{0, 0, d->w, d->h}, dstReq);  // dsttex.sample_bounds(dstReq)
  db = IRect{db.x0 - dstReq.x0, db.y0 - dstReq.y0, db.x1 - dstReq.x0, db.y1 - dstReq.y0};
  db = irect_intersect(db, clip);
  if (db.x1 <= db.x0 || db.y1 <= db.y0) return WRCU_OK;
  YuvBlitArgs a;
  memset(&a, 0, sizeof a);
  // linear_convert_yuv's float set-up, step for step (fp32, no contraction)
  volatile float su = (float)srcReq.x0, sv = (float)srcReq.y0;
  volatile float du = (float)sr[2] / (float)dr[2], dv = (float)sr[3] / (float)dr[3];
  if (flip_x) { su = su + (float)sr[2]; du = -du; }
  if (flip_y) { sv = sv + (float)sr[3]; dv = -dv; }
  { volatile float t = du * ((float)db.x0 + 0.5f); su = su + t; }
  { volatile float t = dv * ((float)db.y0 + 0.5f); sv = sv + t; }
  volatile float csx = (float)tu->w / (float)ty->w, csy = (float)tu->h / (float)ty->h;
  volatile float cu = su * csx, cv = sv * csy, cdu = du * csx, cdv = dv * csy;
  const float qoff = 0.5f - 0.5f * 128.0f;  // linearQuantize(P, 128) = P * 128 + (0.5 - 0.5 * 128)
  { volatile float t = su * 128.0f; su = t + qoff; } { volatile float t = sv * 128.0f; sv = t + qoff; }
  du = du * 128.0f; dv = dv * 128.0f;
  { volatile float t = cu * 128.0f; cu = t + qoff; } { volatile float t = cv * 128.0f; cv = t + qoff; }
  cdu = cdu * 128.0f; cdv = cdv * 128.0f;
  // linear_row_yuv's row-invariant lanes: cast(init_interp(uv.x, du) * (1 << STEP_BITS)), the per-chunk steps
  volatile float yl = su, cl = cu;
  for (int j = 0; j < 4; j++) {
    { volatile float t = yl * (float)(1 << WR_YUV_STEP_BITS); a.yU0[j] = (int)t; }
    { volatile float t = cl * (float)(1 << WR_YUV_STEP_BITS); a.cU0[j] = (int)t; }
    yl = yl + du;
    cl = cl + cdu;
  }
  { volatile float t = (float)(4 << WR_YUV_STEP_BITS) * du; a.yDU = (int)t; }
  { volatile float t = (float)(4 << WR_YUV_STEP_BITS) * cdu; a.cDU = (int)t; }
  a.v0 = sv; a.dv = dv; a.cv0 = cv; a.cdv = cdv;
  a.span = db.x1 - db.x0;
  a.rows = db.y1 - db.y0;
  // the half-resolution fast path (composite.h:1089-1123): chunks before it, pixels inside it; 8-bit planes only
  a.fast = r8 && a.yDU >= a.cDU && a.cDU > 0 && a.yDU <= (4 << (WR_YUV_STEP_BITS + 7)) && a.cDU <= (2 << (WR_YUV_STEP_BITS + 7));
  if (a.fast) {
    int span = a.span, yx = a.yU0[0], cx = a.cU0[0];
    while ((yx < 0 || cx < 0) && span >= 4) { span -= 4; yx += a.yDU; cx += a.cDU; a.pre++; }
    const int in_y = (((ty->w - 4) << (WR_YUV_STEP_BITS + 7)) - yx) / a.yDU, in_c = (((tu->w - 4) << (WR_YUV_STEP_BITS + 7)) - cx) / a.cDU;
    int inside = (in_y < in_c ? in_y : in_c) * 4;
    if (inside > (span & ~3)) inside = span & ~3;
    a.inside = inside > 0 ? inside : 0;
  }
  a.dst = d->dptr; a.dst_pitch = (int)d->pitch;
  a.dx = dstReq.x0 + db.x0; a.dy = dstReq.y0 + db.y0;
  a.yp = ty->dptr; a.up = tu->dptr; a.vp = tv->dptr;
  a.y_pitch = (int)ty->pitch; a.c_pitch = (int)tu->pitch;
  a.yw = ty->w; a.yh = ty->h; a.cw = tu->w; a.ch = tu->h;
  a.color_space = color_space;
  a.rescale_bits = r16 ? (int)color_depth - 1 - 8 : 0;
#ifdef WRCU_HOSTEMU
  if (r16) wr_sw_composite_blit_yuv16(a);
  else wr_sw_composite_blit_yuv(a);
#else
  const int chunks = (a.span + 3) / 4;
  dim3 block(32, 4), grid((unsigned)((chunks + 31) / 32), (unsigned)((a.rows + 3) / 4));
  if (r16) wr_sw_composite_blit_yuv16<<<grid, block, 0, c->stream>>>(a);
  else wr_sw_composite_blit_yuv<<<grid, block, 0, c->stream>>>(a);
  WRCU_CUDA(c, cudaGetLastError());
#endif
  c->stats.kernel_launches++;
  return WRCU_OK;
}

// ---- multi-GPU: shared framebuffer + stream-ordered flags (SURVEY.md §8e) -----------------------
#ifdef WRCU_HOSTEMU
static uint64_t wr_pid() { return 1; }
#else
#include <unistd.h>
static uint64_t wr_pid() { return (uint64_t)getpid(); }
__global__ void wr_flag_signal(uint32_t* flag, uint32_t value) {
  __threadfence_system();  // (the stores of earlier kernels are already performed at their completion)
  *(volatile uint32_t*)flag = value;
  __threadfence_system();
}
__global__ void wr_flag_wait(const uint32_t* flag, uint32_t value, int* timeout_counter) {
  unsigned long long t0, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if ((int32_t)(v - value) >= 0) return;
    __nanosleep(200);
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t - t0 > 2000000000ull) {  // 2 s: the peer is gone; do not hold the GPU
      atomicAdd(timeout_counter, 1 << 20);
      return;
    }
  }
}
#endif
// In-process peers (several contexts driven by one process): a signal is also recorded as a CUDA event, and
// a wait that is queued after it takes the event instead of the polling kernel.  Two streams of one process
// may share a hardware work queue, and a polling kernel at the head of that queue would keep the very
// signal it waits for from starting (until its 2 s timeout); events are ordered by the driver.  Contexts in
// different processes (one rank per GPU) only ever wait on flags written from another device.
#ifndef WRCU_HOSTEMU
#include <map>
#include <mutex>
struct WrSigRec { cudaEvent_t ev; uint32_t value; int device; };
static std::mutex g_sig_mu;
static std::map<uintptr_t, WrSigRec> g_sig;
static void sig_forget(const uint32_t* base, int count) {
  std::lock_guard<std::mutex> lk(g_sig_mu);
  for (int i = 0; i < count; i++) {
    auto it = g_sig.find((uintptr_t)(base + i));
    if (it == g_sig.end()) continue;
    cudaEventDestroy(it->second.ev);
    g_sig.erase(it);
  }
}
#endif
// make `dev` reachable from this context's device
static int enable_peer(wrcu_ctx* c, int dev) {
#ifndef WRCU_HOSTEMU
  if (dev == c->device) return WRCU_OK;
  int can = 0;
  WRCU_CUDA(c, cudaDeviceCanAccessPeer(&can, c->device, dev));
  if (!can) return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "device %d cannot access device %d", c->device, dev);
  cudaError_t e = cudaDeviceEnablePeerAccess(dev, 0);
  if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
    return wrcu_fail(c, WRCU_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
  cudaGetLastError();
#endif
  return WRCU_OK;
}

extern "C" int wrcu_texture_export(wrcu_ctx* c, wrcu_tex id, wrcu_ipc_texture* out) {
  WrTexture* t = get_tex(c, id);
  if (!t || !out || t->imported) return wrcu_fail(c, WRCU_ERR_INVALID, "texture_export: bad arguments");
  cudaSetDevice(c->device);
  memset(out, 0, sizeof *out);
#ifndef WRCU_HOSTEMU
  static_assert(sizeof(cudaIpcMemHandle_t) <= sizeof out->handle, "ipc handle size");
  cudaIpcMemHandle_t h;
  WRCU_CUDA(c, cudaIpcGetMemHandle(&h, t->dptr));
  memcpy(out->handle, &h, sizeof h);
#endif
  out->pid = wr_pid();
  out->address = (uint64_t)(uintptr_t)t->dptr;
  out->pitch = t->pitch;
  out->format = t->fmt; out->width = t->w; out->height = t->h; out->device = c->device;
  return WRCU_OK;
}

extern "C" int wrcu_texture_import(wrcu_ctx* c, const wrcu_ipc_texture* in, wrcu_tex* out) {
  if (!in || !out || !fmt_bpp(in->format) || in->width <= 0 || in->height <= 0)
    return wrcu_fail(c, WRCU_ERR_INVALID, "texture_import: bad arguments");
  cudaSetDevice(c->device);
  void* p = nullptr;
  bool ipc = false;
  if (in->pid == wr_pid()) {
    int rc = enable_peer(c, in->device);
    if (rc != WRCU_OK) return rc;
    p = (void*)(uintptr_t)in->address;
  } else {
#ifndef WRCU_HOSTEMU
    cudaIpcMemHandle_t h;
    memcpy(&h, in->handle, sizeof h);
    WRCU_CUDA(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ipc = true;
#else
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "texture_import: no IPC in the host emulation");
#endif
  }
  for (int i = 1; i < wrcu_ctx::MAX_TEX; i++) {
    if (c->tex[i].live) continue;
    WrTexture& t = c->tex[i];
    t = WrTexture();
    t.fmt = in->format; t.w = in->width; t.h = in->height; t.bpp = fmt_bpp(in->format);
    t.pitch = (size_t)in->pitch;
    t.dptr = (uint8_t*)p;
    t.imported = true;
    t.ipc_mapped = ipc;
    t.live = true;
    make_tensor_map(c, i);
    *out = (wrcu_tex)i;
    return WRCU_OK;
  }
  return wrcu_fail(c, WRCU_ERR_OOM, "texture_import: out of texture handles");
}

extern "C" int wrcu_peer_flags_create(wrcu_ctx* c, int count, wrcu_ipc_flags* out) {
  if (!out || count <= 0 || count > 4096 || c->flags) return wrcu_fail(c, WRCU_ERR_INVALID, "peer_flags_create: bad arguments");
  cudaSetDevice(c->device);
  WRCU_CUDA(c, cudaMalloc((void**)&c->flags, (size_t)count * 4));
  // zeroed before anyone can signal: the legacy-stream cudaMemset does not order against other contexts' streams
  WRCU_CUDA(c, cudaMemsetAsync(c->flags, 0, (size_t)count * 4, c->stream));
  WRCU_CUDA(c, cudaStreamSynchronize(c->stream));
  c->n_flags = count;
  memset(out, 0, sizeof *out);
#ifndef WRCU_HOSTEMU
  cudaIpcMemHandle_t h;
  WRCU_CUDA(c, cudaIpcGetMemHandle(&h, c->flags));
  memcpy(out->handle, &h, sizeof h);
#endif
  out->pid = wr_pid();
  out->address = (uint64_t)(uintptr_t)c->flags;
  out->count = count;
  out->device = c->device;
  return WRCU_OK;
}

extern "C" int wrcu_peer_flags_open(wrcu_ctx* c, const wrcu_ipc_flags* in, int* peer_id) {
  if (!in || !peer_id || in->count <= 0) return wrcu_fail(c, WRCU_ERR_INVALID, "peer_flags_open: bad arguments");
  cudaSetDevice(c->device);
  wrcu_ctx::PeerFlags pf = {nullptr, in->count, false};
  if (in->pid == wr_pid()) {
    int rc = enable_peer(c, in->device);
    if (rc != WRCU_OK) return rc;
    pf.ptr = (uint32_t*)(uintptr_t)in->address;
  } else {
#ifndef WRCU_HOSTEMU
    cudaIpcMemHandle_t h;
    memcpy(&h, in->handle, sizeof h);
    void* p = nullptr;
    WRCU_CUDA(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    pf.ptr = (uint32_t*)p;
    pf.ipc = true;
#else
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "peer_flags_open: no IPC in the host emulation");
#endif
  }
  c->peers.push_back(pf);
  *peer_id = (int)c->peers.size() - 1;
  return WRCU_OK;
}

extern "C" int wrcu_peer_signal(wrcu_ctx* c, int peer_id, int slot, uint32_t value) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  if (peer_id < 0 || peer_id >= (int)c->peers.size() || slot < 0 || slot >= c->peers[peer_id].count)
    return wrcu_fail(c, WRCU_ERR_INVALID, "peer_signal: bad arguments");
  cudaSetDevice(c->device);
#ifndef WRCU_HOSTEMU
  wr_flag_signal<<<1, 1, 0, c->stream>>>(c->peers[peer_id].ptr + slot, value);
  c->stats.kernel_launches++;
  WRCU_CUDA(c, cudaGetLastError());
  if (!c->peers[peer_id].ipc) {
    std::lock_guard<std::mutex> lk(g_sig_mu);
    WrSigRec& r = g_sig[(uintptr_t)(c->peers[peer_id].ptr + slot)];
    if (!r.ev) {
      WRCU_CUDA(c, cudaEventCreateWithFlags(&r.ev, cudaEventDisableTiming));
      r.device = c->device;
    }
    if (r.device == c->device) {  // (an event is recorded on streams of the device it was created on)
      WRCU_CUDA(c, cudaEventRecord(r.ev, c->stream));
      r.value = value;
    }
  }
#else
  c->peers[peer_id].ptr[slot] = value;
#endif
  return WRCU_OK;
}

extern "C" int wrcu_peer_wait(wrcu_ctx* c, int slot, uint32_t value) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  if (!c->flags || slot < 0 || slot >= c->n_flags) return wrcu_fail(c, WRCU_ERR_INVALID, "peer_wait: bad arguments");
  cudaSetDevice(c->device);
#ifndef WRCU_HOSTEMU
  {
    std::lock_guard<std::mutex> lk(g_sig_mu);
    auto it = g_sig.find((uintptr_t)(c->flags + slot));
    if (it != g_sig.end() && it->second.ev && (int32_t)(it->second.value - value) >= 0) {
      WRCU_CUDA(c, cudaStreamWaitEvent(c->stream, it->second.ev, 0));
      c->n_wait_event++;
      return WRCU_OK;
    }
  }
  wr_flag_wait<<<1, 1, 0, c->stream>>>(c->flags + slot, value, c->dev_err);
  c->n_wait_kernel++;
  c->stats.kernel_launches++;
  WRCU_CUDA(c, cudaGetLastError());
#endif
  return WRCU_OK;
}

// ---- frame ---------------------------------------------------------------------------
extern "C" int wrcu_frame_begin(wrcu_ctx* c, const wrcu_frame_tables* t) {
  if (!t) return wrcu_fail(c, WRCU_ERR_INVALID, "frame_begin: null tables");
  cudaSetDevice(c->device);
  { int rcf = flush_pending(c); if (rcf != WRCU_OK) return rcf; }
  // Uploads and GPU-cache updates issued since the last wrcu_frame_end (Renderer::render runs
  // update_texture_cache / update_gpu_cache before draw_frame) were staged into the outgoing arena
  // AFTER its `done` event was recorded: re-record it so the next reuse of that arena waits for them
  // too.  (Also covers arena 0 before the very first frame.)
  {
    Arena* out = &c->arena[c->cur_arena];
    if (out->used > 0) {
      WRCU_CUDA(c, cudaEventRecord(out->done, c->stream));
      out->in_flight = true;
    }
  }
  // switch arena; wait until the frame that last used it has drained
  c->cur_arena ^= 1;
  Arena* a = &c->arena[c->cur_arena];
  if (a->in_flight) {
    WRCU_CUDA(c, cudaEventSynchronize(a->done));
    a->in_flight = false;
  }
  a->used = 0;
  // all seven tables travel in ONE host-to-device copy (they are a few KB each)
  struct TabDesc { const void* src; size_t texels; size_t off; };
  TabDesc td[7] = {{t->prim_headers_f, t->prim_headers_f_texels, 0}, {t->prim_headers_i, t->prim_headers_i_texels, 0},
                   {t->transforms, t->transforms_texels, 0},         {t->render_tasks, t->render_tasks_texels, 0},
                   {t->gpu_cache, t->gpu_cache_texels, 0},           {t->gpu_buffer_f, t->gpu_buffer_f_texels, 0},
                   {t->gpu_buffer_i, t->gpu_buffer_i_texels, 0}};
  size_t total = 0;
  for (int i = 0; i < 7; i++) {
    if (td[i].texels && !td[i].src) return wrcu_fail(c, WRCU_ERR_INVALID, "frame_begin: null table %d", i);
    td[i].off = total;
    total += (td[i].texels * 16 + 255) & ~(size_t)255;
  }
  uint8_t* dbase = nullptr;
  c->tables = FrameTablesDev();  // last frame's pointers must not be rebased if the arena grows below
  if (total) {
    size_t off = 0;
    int rc = arena_reserve(c, total, &off);
    if (rc != WRCU_OK) return rc;
    for (int i = 0; i < 7; i++)
      if (td[i].texels) memcpy(a->host + off + td[i].off, td[i].src, td[i].texels * 16);
    mark_dirty(c, off, off + total);  // copied with the first submission's instances (flush_pending)
    c->stats.h2d_bytes += total;
    dbase = a->dev + off;
  }
#define TAB(i, field, T)                                                         \
  c->tables.n_##field = (int)td[i].texels;                                        \
  c->tables.field = td[i].texels ? (const T*)(dbase + td[i].off) : nullptr;
  TAB(0, prim_headers_f, float4)
  TAB(1, prim_headers_i, int4)
  TAB(2, transforms, float4)
  TAB(3, render_tasks, float4)
  TAB(4, gpu_cache, float4)
  TAB(5, gpu_buffer_f, float4)
  TAB(6, gpu_buffer_i, int4)
#undef TAB
  c->gpu_cache_bound = false;
  if (!t->gpu_cache && !t->gpu_cache_texels && c->gpu_cache_dev) {
    // the persistent GPU cache texture maintained by wrcu_gpu_cache_update
    c->tables.gpu_cache = c->gpu_cache_dev;
    c->tables.n_gpu_cache = c->gpu_cache_rows * 1024;
    c->gpu_cache_bound = true;
  }
  return WRCU_OK;
}

extern "C" int wrcu_frame_end(wrcu_ctx* c) {
  cudaSetDevice(c->device);
  { int rcf = flush_pending(c); if (rcf != WRCU_OK) return rcf; }
  Arena* a = &c->arena[c->cur_arena];
  WRCU_CUDA(c, cudaEventRecord(a->done, c->stream));
  a->in_flight = true;
  return WRCU_OK;
}

// ---- targets -------------------------------------------------------------------------
extern "C" int wrcu_target_bind(wrcu_ctx* c, wrcu_tex color, wrcu_tex depth, const float projection[16],
                                const int32_t viewport[4]) {
  WrTexture* t = get_tex(c, color);
  if (!t || (t->fmt != WRCU_FMT_RGBA8 && t->fmt != WRCU_FMT_R8) || !projection || !viewport)
    return wrcu_fail(c, WRCU_ERR_INVALID, "target_bind: bad colour target");
  if (depth) {
    WrTexture* d = get_tex(c, depth);
    if (!d || d->fmt != WRCU_FMT_DEPTH24 || d->w != t->w || d->h != t->h)
      return wrcu_fail(c, WRCU_ERR_INVALID, "target_bind: bad depth target");
  }
  if (t->pending_read) {  // an async readback of this texture must finish before it is drawn to again
    cudaSetDevice(c->device);
    int rc = wait_fence(c, t->pending_read, true);
    if (rc != WRCU_OK) return rc;
    t->pending_read = 0;
  }
  c->color_tex = color;
  c->depth_tex = depth;
  memcpy(c->proj, projection, sizeof c->proj);
  memcpy(c->vp, viewport, sizeof c->vp);
  return WRCU_OK;
}

static inline int host_round_pixel(float v) { return (int)(v * 255.0f + 0.5f); }

// A texture with an asynchronous readback in flight must not be written before the copy has read it
// (hosts that cache their target binding skip wrcu_target_bind, so draws and clears check as well).
static int wait_pending_read(wrcu_ctx* c, WrTexture* t) {
  if (!t || !t->pending_read) return WRCU_OK;
  int rc = wait_fence(c, t->pending_read, true);
  if (rc == WRCU_OK) t->pending_read = 0;
  return rc;
}

extern "C" int wrcu_clear(wrcu_ctx* c, const int32_t rect[4], const float color[4], const float* depth) {
  WrTexture* t = get_tex(c, c->color_tex);
  if (!t) return wrcu_fail(c, WRCU_ERR_INVALID, "clear: no target bound");
  cudaSetDevice(c->device);
  { int rcw = wait_pending_read(c, t); if (rcw != WRCU_OK) return rcw; }
  int x0 = 0, y0 = 0, x1 = t->w, y1 = t->h;
  if (rect) {
    x0 = rect[0] > 0 ? rect[0] : 0;
    y0 = rect[1] > 0 ? rect[1] : 0;
    x1 = rect[0] + rect[2] < t->w ? rect[0] + rect[2] : t->w;
    y1 = rect[1] + rect[3] < t->h ? rect[1] + rect[3] : t->h;
  }
  if (x1 <= x0 || y1 <= y0) return WRCU_OK;
  // queued in order with the batches (flush_pending): a clear between two batches of a submission must stay there
  PendingOp op;
  op.type = 0;
  op.cx0 = x0; op.cy0 = y0; op.cx1 = x1; op.cy1 = y1;
  if (color) {
    // ClearTexSubImage: round_pixel, truncating U8 convert, BGRA swizzle (gl.cc:2426-2481)
    uint32_t r = host_round_pixel(color[0]) & 0xFF, g = host_round_pixel(color[1]) & 0xFF;
    uint32_t b = host_round_pixel(color[2]) & 0xFF, a = host_round_pixel(color[3]) & 0xFF;
    op.c_ptr = t->dptr; op.c_pitch = (int)t->pitch; op.c_fmt = t->fmt;
    op.c_val = t->fmt == WRCU_FMT_RGBA8 ? (b | (g << 8) | (r << 16) | (a << 24)) : r;
  }
  if (depth && c->depth_tex) {
    WrTexture* d = get_tex(c, c->depth_tex);
    op.d_ptr = d->dptr; op.d_pitch = (int)d->pitch;
    op.d_val = (uint32_t)((double)*depth * 0xFFFFFF);  // gl.cc:2391
  }
  if (!op.c_ptr && !op.d_ptr) return WRCU_OK;
  pending(c).push_back(op);
  if (pending(c).size() >= (size_t)wrcu_ctx::QMAX || c->immediate) return flush_pending(c);
  return WRCU_OK;
}

static int launch_clear(wrcu_ctx* c, const PendingOp& op) {
  dim3 grid((unsigned)((op.cx1 - op.cx0 + 1023) / 1024), (unsigned)(op.cy1 - op.cy0));
  if (grid.x > 8) grid.x = 8;
  if (op.c_ptr) {
    if (op.c_fmt == WRCU_FMT_RGBA8)
      WR_LAUNCH(wr_clear_u32, grid, 256, c->launch_stream, op.c_ptr, op.c_pitch, op.cx0, op.cy0, op.cx1, op.cy1, op.c_val);
    else
      WR_LAUNCH(wr_clear_u8, grid, 256, c->launch_stream, op.c_ptr, op.c_pitch, op.cx0, op.cy0, op.cx1, op.cy1, (uint8_t)op.c_val);
    c->stats.kernel_launches++;
  }
  if (op.d_ptr) {
    WR_LAUNCH(wr_clear_u32, grid, 256, c->launch_stream, op.d_ptr, op.d_pitch, op.cx0, op.cy0, op.cx1, op.cy1, op.d_val);
    c->stats.kernel_launches++;
  }
  WRCU_CUDA(c, cudaGetLastError());
  return WRCU_OK;
}

// ---- draws ---------------------------------------------------------------------------
static TexView tex_view(wrcu_ctx* c, wrcu_tex id) {
  TexView v;
  memset(&v, 0, sizeof v);
  WrTexture* t = get_tex(c, id);
  if (!t) {
    v.w = v.h = 1;  // null sampler (gl.cc:894-905); ptr stays null → callers check
    return v;
  }
  v.ptr = t->dptr;
  v.w = t->w;
  v.h = t->h;
  v.pitch = (int)t->pitch;
  v.filter = t->w >= 2 ? t->filter : WRCU_NEAREST;  // init_filter, gl.cc:870-877
  v.fmt = t->fmt;
  v.tmap_id = t->has_tmap ? t->tmap_slot : 0;
  return v;
}

static int ensure_cmd_capacity(wrcu_ctx* c, size_t n) {
  if (n <= c->cmd_cap) return WRCU_OK;
  WRCU_CUDA(c, cudaStreamSynchronize(c->stream));
  if (c->cmd_hot) cudaFree(c->cmd_hot);
  if (c->cmd_cold) cudaFree(c->cmd_cold);
  c->cmd_hot = c->cmd_cold = nullptr;
  size_t cap = align_up(n * 2, 1024);
  WRCU_CUDA(c, cudaMalloc(&c->cmd_hot, cap * sizeof(CmdHot)));
  WRCU_CUDA(c, cudaMalloc(&c->cmd_cold, cap * sizeof(CmdCold)));
  c->cmd_cap = cap;
  return WRCU_OK;
}

static int draw_batch_impl(wrcu_ctx* c, int kind, uint32_t features, const wrcu_draw_state* st,
                           const void* instances, size_t stride, int n, const wrcu_tex* textures);

extern "C" int wrcu_draw_batch(wrcu_ctx* c, int kind, uint32_t features, const wrcu_draw_state* st,
                               const void* instances, size_t stride, int n) {
  return draw_batch_impl(c, kind, features, st, instances, stride, n, nullptr);
}

extern "C" int wrcu_draw_composite_tiles(wrcu_ctx* c, uint32_t features, const wrcu_draw_state* st,
                                         const void* instances, size_t stride, int n, const wrcu_tex* textures) {
  if (!textures) return wrcu_fail(c, WRCU_ERR_INVALID, "draw_composite_tiles: no texture list");
  if (features & WRCU_FEAT_YUV)
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "draw_composite_tiles: YUV surfaces go through wrcu_draw_batch");
  return draw_batch_impl(c, WRCU_KIND_COMPOSITE, features, st, instances, stride, n, textures);
}

#define WR_COPY_MAX_CMDS_HOST 128  // = WR_COPY_MAX_CMDS (shader_composite.cuh): the copy kernel's staged command list
static int draw_batch_impl(wrcu_ctx* c, int kind, uint32_t features, const wrcu_draw_state* st,
                           const void* instances, size_t stride, int n, const wrcu_tex* textures) {
  if (!st || !instances || n < 0 || stride == 0)
    return wrcu_fail(c, WRCU_ERR_INVALID, "draw_batch: bad arguments");
  if (n == 0) return WRCU_OK;
  WrTexture* tgt = get_tex(c, c->color_tex);
  if (!tgt) return wrcu_fail(c, WRCU_ERR_INVALID, "draw_batch: no target bound");
  if (st->blend < 0 || st->blend >= WRCU_BLEND__COUNT)
    return wrcu_fail(c, WRCU_ERR_INVALID, "draw_batch: bad blend key");
  if (st->blend == WRCU_BLEND_SUBPIXEL_DUAL_SOURCE)
    return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "GL dual-source blending: SWGL hosts use the subpixel-text blend override instead");
  cudaSetDevice(c->device);
  { int rcw = wait_pending_read(c, tgt); if (rcw != WRCU_OK) return rcw; }
  c->stats.draw_calls++;
  c->stats.instances += (uint64_t)n;

  int rc;
  size_t views_off = 0;
  if (textures) {
    // one sampler view per instance, staged ahead of the instances
    std::vector<TexView> views((size_t)n);
    for (int i = 0; i < n; i++) {
      views[(size_t)i] = tex_view(c, textures[i]);
      if (!views[(size_t)i].ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "draw_composite_tiles: instance %d has no texture", i);
    }
    void* dviews = nullptr;
    if ((rc = stage(c, views.data(), views.size() * sizeof(TexView), &dviews, false, true)) != WRCU_OK) return rc;
    views_off = (size_t)((uint8_t*)dviews - c->arena[c->cur_arena].dev);
  }
  void* dinst = nullptr;
  if ((rc = stage(c, instances, stride * (size_t)n, &dinst, false, true)) != WRCU_OK) return rc;

  TargetDev T;
  memset(&T, 0, sizeof T);
  T.color = tgt->dptr;
  T.color_pitch = (int)tgt->pitch;
  T.fmt = tgt->fmt;
  T.w = tgt->w;
  T.h = tgt->h;
  WrTexture* dep = (st->depth != WRCU_DEPTH_OFF) ? get_tex(c, c->depth_tex) : nullptr;
  T.depth = dep ? (uint32_t*)dep->dptr : nullptr;
  T.depth_pitch = dep ? (int)dep->pitch : 0;
  memcpy(T.proj, c->proj, sizeof T.proj);
  memcpy(T.vp, c->vp, sizeof T.vp);
  T.cx0 = 0; T.cy0 = 0; T.cx1 = tgt->w; T.cy1 = tgt->h;
  T.tmap_id = tgt->has_tmap ? tgt->tmap_slot : 0;
  if (st->scissor_enabled) {
    T.cx0 = max(T.cx0, st->scissor[0]);
    T.cy0 = max(T.cy0, st->scissor[1]);
    T.cx1 = min(T.cx1, st->scissor[0] + st->scissor[2]);
    T.cy1 = min(T.cy1, st->scissor[1] + st->scissor[3]);
  }

  if (T.cx1 <= T.cx0 || T.cy1 <= T.cy0) return WRCU_OK;  // scissor misses the target: SWGL draws nothing

  SetupArgs sa;
  memset(&sa, 0, sizeof sa);
  sa.tgt = T;
  const size_t inst_off = (size_t)((uint8_t*)dinst - c->arena[c->cur_arena].dev);  // pointers are resolved at flush
  sa.stride = (int)stride;
  sa.n = n;
  // (hot / cold / info / pool pointers are assigned when the submission is flushed)
  sa.err_counter = c->dev_err;
  sa.blend_enabled = st->blend != WRCU_BLEND_NONE;
#ifndef WRCU_HOSTEMU
  {
    // Depth runs matter to kinds whose shading depends on the position inside a span (AA ramps, span
    // shader vs fragment tail, interpolated varyings).  Plain solids with blending off never do (their
    // AA / mask flags are dropped, setup_common.cuh wr_emit_quad).
    bool kind_runs = false;
    switch (kind) {
      case WRCU_KIND_BRUSH_SOLID: kind_runs = st->blend != WRCU_BLEND_NONE; break;
      case WRCU_KIND_QUAD_TEXTURED: case WRCU_KIND_BRUSH_IMAGE: case WRCU_KIND_BRUSH_LINEAR_GRADIENT:
      case WRCU_KIND_BRUSH_BLEND: case WRCU_KIND_BRUSH_MIX_BLEND: case WRCU_KIND_BRUSH_OPACITY: case WRCU_KIND_TEXT_RUN:
      case WRCU_KIND_BRUSH_YUV_IMAGE: case WRCU_KIND_QUAD_RADIAL_GRADIENT: case WRCU_KIND_QUAD_CONIC_GRADIENT:
      case WRCU_KIND_SPLIT_COMPOSITE:
        kind_runs = true; break;
      default: break;
    }
    if (kind_runs && T.depth) {
      if (!c->fail_pool) {
        c->fail_cap = 16 << 20;  // 64 MiB of bitmaps per batch; commands beyond it keep span-relative phase
        if (cudaMalloc((void**)&c->fail_pool, (size_t)c->fail_cap * 4) != cudaSuccess) {
          c->fail_pool = nullptr;
          c->fail_cap = 0;
          cudaGetLastError();
        }
      }
      if (c->fail_pool) {
        sa.depth_runs = 1;
        sa.fail_cap = c->fail_cap;
      }
    }
  }
#endif
  // draw_perspective (w differs between an instance's vertices): the kinds whose fragment stage carries the
  // per-sample 1/w path; the solid colour case of ps_quad_textured shares brush_solid's shader
  sa.persp_ok = kind == WRCU_KIND_BRUSH_SOLID || kind == WRCU_KIND_SPLIT_COMPOSITE || kind == WRCU_KIND_QUAD_TEXTURED ||
                kind == WRCU_KIND_BRUSH_OPACITY || kind == WRCU_KIND_BRUSH_BLEND || kind == WRCU_KIND_BRUSH_MIX_BLEND ||
                (kind == WRCU_KIND_BRUSH_IMAGE && !(features & WRCU_FEAT_REPETITION));
  // copy class (shader_composite.cuh): 1 = 1:1 tile copies and solid fills, 2 = fills only (the clear tile's dest-out)
  sa.copy_ok = T.depth ? 0 : (st->blend == WRCU_BLEND_NONE || st->blend == WRCU_BLEND_PREMULTIPLIED_ALPHA) ? 1
                             : st->blend == WRCU_BLEND_PREMULTIPLIED_DEST_OUT ? 2 : 0;
  if (kind == WRCU_KIND_COMPOSITE && sa.copy_ok && !(features & WRCU_FEAT_YUV)) {
    // The copy kernel moves boxes of different instances concurrently: a batch whose instances overlap keeps
    // the ordered tile kernel.  Picture-cache tiles never overlap; checked here on the host copies of the
    // CompositeInstance rects (device rect ∩ clip rect, rounded outwards), n is a tile list's length.
    if (n > WR_COPY_MAX_CMDS_HOST || stride < 32) sa.copy_ok = 0;
    else {
      std::vector<float> bb((size_t)n * 4);
      for (int i = 0; i < n; i++) {
        const float* f = (const float*)((const uint8_t*)instances + (size_t)i * stride);
        const float x0 = fminf(f[0], f[2]), x1 = fmaxf(f[0], f[2]), y0 = fminf(f[1], f[3]), y1 = fmaxf(f[1], f[3]);
        bb[4 * i + 0] = floorf(fmaxf(x0, f[4])); bb[4 * i + 1] = floorf(fmaxf(y0, f[5]));
        bb[4 * i + 2] = ceilf(fminf(x1, f[6]));  bb[4 * i + 3] = ceilf(fminf(y1, f[7]));
      }
      for (int i = 0; i < n && sa.copy_ok; i++) {
        if (bb[4 * i + 2] <= bb[4 * i] || bb[4 * i + 3] <= bb[4 * i + 1]) continue;
        for (int j = 0; j < i; j++)
          if (bb[4 * j] < bb[4 * i + 2] && bb[4 * i] < bb[4 * j + 2] && bb[4 * j + 1] < bb[4 * i + 3] && bb[4 * i + 1] < bb[4 * j + 3] &&
              bb[4 * j + 2] > bb[4 * j] && bb[4 * j + 3] > bb[4 * j + 1]) { sa.copy_ok = 0; break; }
      }
    }
  }
  sa.color0 = tex_view(c, st->color[0]);
  sa.color1 = tex_view(c, st->color[1]);
  sa.color2 = tex_view(c, st->color[2]);
  if (textures) sa.color0 = tex_view(c, textures[0]);  // (sa.tex_list: resolved from views_off at flush)
  size_t bin_need = 0;
  // Bitmask bins for batches with many instances: the per-tile command scan of the raster
  // kernel costs tiles x n hot records of L2 traffic; with bins it reads n/32 words per tile.
  {
    const int tiles_x = (T.w + WRCU_TILE_W - 1) / WRCU_TILE_W, tiles_y = (T.h + WRCU_TILE_H - 1) / WRCU_TILE_H;
    const size_t words = ((size_t)n + 31) / 32;
    const size_t any_words = ((size_t)tiles_x * tiles_y + 31) / 32;
    const size_t need = ((size_t)tiles_x * tiles_y + 1) * words + 2 * any_words + 1;  // + the wide mask + the tile-any bitmap
                                                                                         // + the ordered-tile bitmap (text)
    if (n >= 512 && need * 4 <= (size_t)96 << 20) {
      // pointers into the submission's bin area are assigned at flush (PendingOp::bin_need)
      bin_need = need;
      sa.bin_words = (int)words;
      sa.bin_tiles_x = tiles_x;
      sa.any_words = (int)any_words;
    }
  }
  sa.clip_mask = tex_view(c, st->clip_mask);

  int sblocks = (n + 127) / 128;
#ifndef WRCU_HOSTEMU
  if (n <= 64) {  // small batch: a warp per instance (setup_common.cuh WR_SETUP_KERNEL)
    sa.warp_per_inst = 1;
    sblocks = (n * 32 + 127) / 128;
  }
#endif
  switch (kind) {
    case WRCU_KIND_QUAD_TEXTURED:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "quad instance stride < 16");
      /* set-up: wr_setup_quad_textured, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_SOLID:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      /* set-up: wr_setup_brush_solid, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_IMAGE:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (features & WRCU_FEAT_DUAL_SOURCE_BLENDING)
        return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "brush_image DUAL_SOURCE_BLENDING variant not built (SWGL does not build it either)");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "brush_image without sColor0");
      sa.features = features;
      /* set-up: wr_setup_brush_image, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_LINEAR_GRADIENT:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      sa.features = features;
      /* set-up: wr_setup_brush_linear_gradient, run by flush_pending */;
      break;
    case WRCU_KIND_TEXT_RUN:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "ps_text_run without sColor0");
      sa.features = features;
      /* set-up: wr_setup_text_run, run by flush_pending */;
      break;
    case WRCU_KIND_QUAD_MASK:
      if (stride < 32) return wrcu_fail(c, WRCU_ERR_INVALID, "MaskInstance stride < 32");
      sa.features = features;
      /* set-up: wr_setup_quad_mask, run by flush_pending */;
      break;
    case WRCU_KIND_CLIP_RECTANGLE:
      if (stride < 200) return wrcu_fail(c, WRCU_ERR_INVALID, "ClipMaskInstanceRect stride < 200");
      sa.features = features;
      /* set-up: wr_setup_clip_rectangle, run by flush_pending */;
      break;
    case WRCU_KIND_SCALE:
      if (stride < 36) return wrcu_fail(c, WRCU_ERR_INVALID, "ScalingInstance stride < 36");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "cs_scale without sColor0");
      sa.features = features;
      /* set-up: wr_setup_scale, run by flush_pending */;
      break;
    case WRCU_KIND_QUAD_RADIAL_GRADIENT:
    case WRCU_KIND_QUAD_CONIC_GRADIENT:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      sa.features = features;
      sa.kind = kind;
      /* set-up: wr_setup_quad_gradient, run by flush_pending */;
      break;
    case WRCU_KIND_LINE_DECORATION:
      if (stride < 36) return wrcu_fail(c, WRCU_ERR_INVALID, "LineDecorationJob stride < 36");
      sa.features = features;
      /* set-up: wr_setup_line_decoration, run by flush_pending */;
      break;
    case WRCU_KIND_BORDER_SOLID:
    case WRCU_KIND_BORDER_SEGMENT:
      if (stride < 108) return wrcu_fail(c, WRCU_ERR_INVALID, "BorderInstance stride < 108");
      sa.features = features;
      sa.kind = kind;
      /* set-up: wr_setup_border, run by flush_pending */;
      break;
    case WRCU_KIND_FAST_LINEAR_GRADIENT:
    case WRCU_KIND_LINEAR_GRADIENT:
    case WRCU_KIND_RADIAL_GRADIENT:
    case WRCU_KIND_CONIC_GRADIENT:
      if (stride < (kind == WRCU_KIND_LINEAR_GRADIENT ? 48u : 52u))
        return wrcu_fail(c, WRCU_ERR_INVALID, "gradient task instance stride too small");
      sa.features = features;
      sa.kind = kind;
      /* set-up: wr_setup_cs_gradient, run by flush_pending */;
      break;
    case WRCU_KIND_BLUR:
      if (stride < 24) return wrcu_fail(c, WRCU_ERR_INVALID, "BlurInstance stride < 24");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "cs_blur without sColor0");
      if (!(features & (WRCU_FEAT_ALPHA_TARGET | WRCU_FEAT_COLOR_TARGET)))
        return wrcu_fail(c, WRCU_ERR_INVALID, "cs_blur needs ALPHA_TARGET or COLOR_TARGET");
      sa.features = features;
      /* set-up: wr_setup_blur, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_MIX_BLEND:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (!sa.color0.ptr || !sa.color1.ptr)
        return wrcu_fail(c, WRCU_ERR_INVALID, "brush_mix_blend needs sColor0 (backdrop) and sColor1 (source)");
      sa.features = features;
      /* set-up: wr_setup_brush_mix_blend, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_BLEND:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "brush_blend without sColor0");
      sa.features = features;
      /* set-up: wr_setup_brush_blend, run by flush_pending */;
      break;
    case WRCU_KIND_CLEAR:
      if (stride < 32) return wrcu_fail(c, WRCU_ERR_INVALID, "ClearInstance stride < 32");
      /* set-up: wr_setup_clear, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_OPACITY:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "brush_opacity without sColor0");
      sa.features = features;
      /* set-up: wr_setup_brush_opacity, run by flush_pending */;
      break;
    case WRCU_KIND_SPLIT_COMPOSITE:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (!sa.color0.ptr || sa.color0.fmt != WRCU_FMT_RGBA8)
        return wrcu_fail(c, WRCU_ERR_INVALID, "ps_split_composite needs an RGBA8 surface in sColor0");
      sa.features = features;
      /* set-up: wr_setup_split_composite, run by flush_pending */;
      break;
    case WRCU_KIND_BRUSH_YUV_IMAGE:
      if (stride < 16) return wrcu_fail(c, WRCU_ERR_INVALID, "prim instance stride < 16");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "brush_yuv_image without sColor0");
      sa.features = features;
      /* set-up: wr_setup_brush_yuv_image, run by flush_pending */;
      break;
    case WRCU_KIND_COMPOSITE:
      if (stride < 120) return wrcu_fail(c, WRCU_ERR_INVALID, "CompositeInstance stride < 120");
      if (!sa.color0.ptr) return wrcu_fail(c, WRCU_ERR_INVALID, "composite without sColor0");
      sa.features = features;
      if (features & WRCU_FEAT_YUV) /* set-up: wr_setup_composite_yuv, run by flush_pending */;
      else /* set-up: wr_setup_composite, run by flush_pending */;
      break;
    case WRCU_KIND_CLIP_BOX_SHADOW:
      if (stride < 84) return wrcu_fail(c, WRCU_ERR_INVALID, "ClipMaskInstanceBoxShadow stride < 84");
      if (!sa.color0.ptr || sa.color0.fmt != WRCU_FMT_R8)
        return wrcu_fail(c, WRCU_ERR_INVALID, "cs_clip_box_shadow needs an R8 shadow mask in sColor0");
      sa.features = features;
      /* set-up: wr_setup_clip_box_shadow, run by flush_pending */;
      break;
    default:
      return wrcu_fail(c, WRCU_ERR_UNSUPPORTED, "draw_batch: kind %d not implemented", kind);
  }

  RasterArgs ra;
  memset(&ra, 0, sizeof ra);
  ra.tgt = T;
  ra.n = n;
  ra.blend = st->blend;
  ra.depth_mode = T.depth ? st->depth : WRCU_DEPTH_OFF;
  ra.blend_color = Px{host_round_pixel(st->blend_color[2]) & 0xFFFF, host_round_pixel(st->blend_color[1]) & 0xFFFF,
                      host_round_pixel(st->blend_color[0]) & 0xFFFF, host_round_pixel(st->blend_color[3]) & 0xFFFF};
  ra.color0 = sa.color0;
  ra.color1 = sa.color1;
  ra.color2 = sa.color2;
  ra.bin_words = sa.bin_words;
  ra.any_words = sa.any_words;
  ra.bin_tiles_x = sa.bin_tiles_x;
  ra.tmaps = c->tmaps_dev;
  ra.tmap_acquire = c->tmap_wrapped ? 1 : 0;
  dim3 grid((unsigned)((T.cx1 - 0 + WRCU_TILE_W - 1) / WRCU_TILE_W), (unsigned)((T.cy1 + WRCU_TILE_H - 1) / WRCU_TILE_H));
  if (grid.x == 0 || grid.y == 0) return WRCU_OK;
  // ---- queue the batch: its set-up runs with every other queued batch's in ONE launch (flush_pending) ----
  PendingOp op;
  op.type = 1;
  op.kind = kind;
  op.features = features;
  op.blend = st->blend;
  op.n = n;
  op.sblocks = sblocks;
  op.bin_need = bin_need;
  op.sa = sa;
  op.ra = ra;
  op.inst_off = inst_off;
  op.views_off = textures ? views_off : (size_t)-1;
  if (textures)
    for (int i = 0; i < n; i++) op.tex_reads.push_back(tex_view(c, textures[i]).ptr);
  op.grid_x = grid.x;
  op.grid_y = grid.y;
  pending(c).push_back(op);
  c->pend_instances += (size_t)n;
  if (pending(c).size() >= (size_t)wrcu_ctx::QMAX || c->immediate) return flush_pending(c);
  return WRCU_OK;
}

#ifndef WRCU_HOSTEMU
// A raster-class launch with programmatic stream serialization (see raster.cuh wr_pdl_wait); the ordinary
// launch when the context has it switched off (WRCU_PDL=0).
template <typename K>
static void wr_launch_chain(wrcu_ctx* c, K kernel, unsigned grid, unsigned block, size_t smem, const RasterArgs& ra) {
  // (a launch that directly follows an event wait in its stream is an ordinary one: the programmatic edge is
  // between two kernels, and nothing is gained by leaving it to the driver what an event wait in between means)
  if (!c->pdl || c->plain_next) {
    c->plain_next = false;
    kernel<<<grid, block, smem, c->launch_stream>>>(ra);
    return;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = c->launch_stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, ra);
}
#endif

// The raster launches of one queued batch (its set-up has run): depth-run prepass, then the kernel(s) of its kind.
static int launch_raster(wrcu_ctx* c, PendingOp& op) {
  RasterArgs& ra = op.ra;
  const TargetDev& T = ra.tgt;
  const int kind = op.kind, n = op.n;
  const uint32_t features = op.features;
  dim3 grid(op.grid_x, op.grid_y);
  // Device-side dispatch: the setup kernel decides whether the whole batch is
  // plain solid quads; the specialised and the generic kernel each return at
  // once when it is not their turn (the host never has to wait for the flag).
#ifndef WRCU_HOSTEMU
  if (op.sa.depth_runs) {
    // depth runs: the failing-sample bitmaps of this batch, before any of its depth writes
    ra.fail_pool = c->fail_pool;
    // grid: a CTA per command in the command-major mode (n >= 48, see the kernel), else row groups over the chip —
    // a quarter of it when other render targets' kernels share the GPU (side streams)
    int fgrid = c->sm_count * 4;
    if (n >= 48) fgrid = n < fgrid ? n : fgrid;
    else if (c->side_reduce) fgrid = c->sm_count * c->side_ctas_per_sm;
    wr_depth_fail_rows<<<fgrid, 256, 0, c->launch_stream>>>(ra, c->fail_pool);
    c->stats.kernel_launches++;
  }
#endif
  if (c->profile) WRCU_CUDA(c, cudaEventRecord(c->p0, c->launch_stream));
  bool fast_ok = T.fmt == WRCU_FMT_RGBA8 && op.blend == WRCU_BLEND_PREMULTIPLIED_ALPHA &&
                 ra.depth_mode == WRCU_DEPTH_OFF &&
                 (kind == WRCU_KIND_QUAD_TEXTURED || kind == WRCU_KIND_BRUSH_SOLID);  // the only kinds that emit CMD_CONST_COLOR
  ra.fast_eligible = fast_ok ? 1 : 0;
  if (fast_ok) {
#ifdef WRCU_HOSTEMU
    wr_raster_solid_premult(ra);
#else
    // persistent CTAs: size the grid so the tile count splits evenly over the
    // CTAs resident at once (a partial last wave would idle most of the chip)
    if (c->fast_ctas_per_sm == 0) {
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, wr_raster_solid_premult, FAST_THREADS, 0) != cudaSuccess || nb < 1)
        nb = 8;
      c->fast_ctas_per_sm = nb;
    }
    if (n <= c->flat_max) {
      // shallow batch: the streaming variant (8 pixels per thread over the bounding box; grid sized for the
      // whole target, threads beyond the box leave at once)
      const long long groups = ((long long)(T.w + 3) / 4) * ((T.h + 1) / 2);
      long long blocks = (groups + FLAT_THREADS - 1) / FLAT_THREADS;
      const long long cap = (long long)c->sm_count * 64;
      if (blocks > cap) blocks = cap;
      wr_launch_chain(c, wr_raster_solid_flat, (unsigned)blocks, FLAT_THREADS, 0, ra);
    } else {
    const int n_tiles = (int)(grid.x * grid.y);
    const int sms = c->sm_count > 0 ? c->sm_count : 148;
    int best_grid = n_tiles;
    if (n_tiles > sms * c->fast_ctas_per_sm) {
      double best_eff = 0.0;
      for (int k = c->fast_ctas_per_sm; k >= max(1, c->fast_ctas_per_sm / 2); k--) {
        const int slots = sms * k;
        const int rounds = (n_tiles + slots - 1) / slots;
        const double eff = (double)n_tiles / ((double)rounds * slots);
        if (eff > best_eff + 1e-9) { best_eff = eff; best_grid = slots; }
      }
    }
    wr_launch_chain(c, wr_raster_solid_premult, (unsigned)best_grid, FAST_THREADS, 0, ra);
    }
#endif
    c->stats.kernel_launches++;
  }
  // generic kernels: persistent CTAs over the batch's tiles; 3 CTAs of 256 threads per SM
  // cover every shader's register budget (<= 128 regs/thread would allow 2; most use 80)
  const int total_tiles = (int)(grid.x * grid.y);
  // On a side stream (several render targets in flight) a small batch takes one persistent CTA per SM instead of
  // three: its CTAs each walk more tiles, but the start-up wave of a 444-CTA launch no longer holds every CTA slot
  // of the chip while most of its CTAs find no tile.
  const int max_ctas = (c->side_reduce && n <= 256) ? c->sm_count * c->side_ctas_per_sm : c->sm_count * 3;
  const int pgrid = total_tiles < max_ctas ? total_tiles : max_ctas;
  // strip mode (raster.cuh WrRowReuse): few commands on a wide target — work items become runs of adjacent tiles,
  // as long as there are still about two items per resident CTA
  ra.strip_seg = 0;
  if (c->strip && n <= 16 && (kind == WRCU_KIND_COMPOSITE || kind == WRCU_KIND_BRUSH_YUV_IMAGE || kind == WRCU_KIND_BRUSH_LINEAR_GRADIENT)) {
    int seg = 10;
    while (seg > 1 && (((int)grid.x + seg - 1) / seg) * (int)grid.y < 2 * max_ctas) seg--;
    if (seg > 1) ra.strip_seg = seg;
  }
#define LAUNCH_RASTER(S)                                                         \
  do {                                                                           \
    auto k_rgba = wr_raster<S, WRCU_FMT_RGBA8>;                                   \
    auto k_r8 = wr_raster<S, WRCU_FMT_R8>;                                        \
    if (T.fmt == WRCU_FMT_RGBA8)                                                 \
      WR_LAUNCH_CHAIN(k_rgba, pgrid, WRCU_THREADS, ra);                          \
    else                                                                         \
      WR_LAUNCH_CHAIN(k_r8, pgrid, WRCU_THREADS, ra);                            \
  } while (0)
  // kinds drawn under depth test: the depth-run variant when this batch has failing-sample bitmaps
#ifdef WRCU_HOSTEMU
#define LAUNCH_RASTER_RUNS(S) LAUNCH_RASTER(S)
#else
#define LAUNCH_RASTER_RUNS(S)                                                    \
  do {                                                                           \
    if (op.sa.depth_runs && T.fmt == WRCU_FMT_RGBA8) {                              \
      auto k_runs = wr_raster<S, WRCU_FMT_RGBA8, true>;                           \
      WR_LAUNCH_CHAIN(k_runs, pgrid, WRCU_THREADS, ra);                          \
    } else LAUNCH_RASTER(S);                                                     \
  } while (0)
#endif
  switch (kind) {
    case WRCU_KIND_CLIP_RECTANGLE: LAUNCH_RASTER(ClipRectShader); break;
    case WRCU_KIND_QUAD_MASK: LAUNCH_RASTER(QuadMaskShader); break;
    case WRCU_KIND_BRUSH_IMAGE:
      if (features & WRCU_FEAT_REPETITION) LAUNCH_RASTER_RUNS(ImageRepeatShader);
      else LAUNCH_RASTER_RUNS(ImageShader);
      break;
    case WRCU_KIND_TEXT_RUN:
#ifndef WRCU_HOSTEMU
      // glyph-major first (a warp per glyph, shader_text.cuh); the tile kernel then draws what it flagged CMD_ORDERED
      if (c->glyph_major && T.fmt == WRCU_FMT_RGBA8 && n >= 8 &&
          (ra.depth_mode == WRCU_DEPTH_OFF || (ra.depth_mode == WRCU_DEPTH_TEST && op.sa.depth_runs))) {
        ra.glyph_major = 1;
        auto k_glyphs = wr_raster_glyphs<WRCU_FMT_RGBA8>;
        const int per_cta = WR_GLYPH_THREADS / 32;
        int ggrid = (n + per_cta - 1) / per_cta;           // persistent warps taking glyphs by ticket
        if (ggrid > c->sm_count * c->glyph_ctas) ggrid = c->sm_count * c->glyph_ctas;
        wr_launch_chain(c, k_glyphs, (unsigned)ggrid, WR_GLYPH_THREADS, 0, ra);
        c->stats.kernel_launches++;
        ra.pdl_early = 0;  // the tile kernel reads what the glyph kernel wrote (flags, BatchInfo::n_ordered)
      }
#endif
      LAUNCH_RASTER_RUNS(TextShader);
      break;
    case WRCU_KIND_BRUSH_LINEAR_GRADIENT: LAUNCH_RASTER_RUNS(GradientShader); break;
    case WRCU_KIND_CLIP_BOX_SHADOW: LAUNCH_RASTER(BoxShadowShader); break;
    case WRCU_KIND_BRUSH_YUV_IMAGE:
      if (ra.color0.fmt == WRCU_FMT_R16) LAUNCH_RASTER_RUNS(CompositeYuv16Shader);
      else LAUNCH_RASTER_RUNS(CompositeYuvShader);
      break;
    case WRCU_KIND_SPLIT_COMPOSITE: LAUNCH_RASTER_RUNS(ImageShader); break;
    case WRCU_KIND_COMPOSITE:
      if (features & WRCU_FEAT_YUV) {
#ifndef WRCU_HOSTEMU
        if (c->yuv_wide && T.fmt == WRCU_FMT_RGBA8 && ra.color0.fmt != WRCU_FMT_R16) { auto k_w = wr_raster<CompositeYuvShaderWide, WRCU_FMT_RGBA8>; WR_LAUNCH_CHAIN(k_w, pgrid, WRCU_THREADS, ra); break; }
#endif
        if (ra.color0.fmt == WRCU_FMT_R16) LAUNCH_RASTER(CompositeYuv16Shader);
        else LAUNCH_RASTER(CompositeYuvShader);
        break;
      }
#ifndef WRCU_HOSTEMU
      if (c->tmaps_dev && T.tmap_id && op.sa.copy_ok) {
        // copy-class tile lists (decided on the device, BatchInfo::all_copy) go through the copy engine;
        // whichever of the two kernels is not in charge returns at once
        const size_t smem0 = (size_t)WR_TMA_STAGES * WR_TMA_BOX_BYTES, smem1 = (size_t)WR_TMA_BLEND_STAGES * 2 * WR_TMA_BOX_BYTES;
        if (!c->copy_attr_set) {
          WRCU_CUDA(c, cudaFuncSetAttribute(wr_composite_copy<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0));
          WRCU_CUDA(c, cudaFuncSetAttribute(wr_composite_copy<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
          c->copy_attr_set = true;
        }
        ra.copy_eligible = 1;
        if (op.blend == WRCU_BLEND_NONE) wr_launch_chain(c, wr_composite_copy<0>, (unsigned)c->sm_count * 3, WR_TMA_THREADS, smem0, ra);
        else if (op.blend == WRCU_BLEND_PREMULTIPLIED_ALPHA) wr_launch_chain(c, wr_composite_copy<1>, (unsigned)c->sm_count * 2, WR_TMA_THREADS, smem1, ra);
        else wr_launch_chain(c, wr_composite_copy<2>, (unsigned)c->sm_count * 2, WR_TMA_THREADS, 0, ra);
        c->stats.kernel_launches++;
      }
#endif
      LAUNCH_RASTER(CompositeShader);
      break;
    case WRCU_KIND_BRUSH_OPACITY: LAUNCH_RASTER_RUNS(OpacityShader); break;
    case WRCU_KIND_BRUSH_BLEND: LAUNCH_RASTER_RUNS(BlendShader); break;
    case WRCU_KIND_BRUSH_MIX_BLEND: LAUNCH_RASTER_RUNS(MixBlendShader); break;
    case WRCU_KIND_BLUR: LAUNCH_RASTER(BlurShader); break;
    case WRCU_KIND_SCALE: LAUNCH_RASTER(ScaleShader); break;
    case WRCU_KIND_FAST_LINEAR_GRADIENT: LAUNCH_RASTER(FastLinearShader); break;
    case WRCU_KIND_LINEAR_GRADIENT: LAUNCH_RASTER(GradientShader); break;
    case WRCU_KIND_RADIAL_GRADIENT: LAUNCH_RASTER(RadialShader); break;
    case WRCU_KIND_CONIC_GRADIENT: LAUNCH_RASTER(ConicShader); break;
    case WRCU_KIND_QUAD_RADIAL_GRADIENT: LAUNCH_RASTER_RUNS(RadialShader); break;
    case WRCU_KIND_QUAD_CONIC_GRADIENT: LAUNCH_RASTER_RUNS(QuadConicShader); break;
    case WRCU_KIND_LINE_DECORATION: LAUNCH_RASTER(LineDecorationShader); break;
    case WRCU_KIND_BORDER_SOLID: LAUNCH_RASTER(BorderSolidShader); break;
    case WRCU_KIND_BORDER_SEGMENT: LAUNCH_RASTER(BorderSegmentShader); break;
    default: LAUNCH_RASTER_RUNS(QuadShader); break;
  }
#undef LAUNCH_RASTER
#undef LAUNCH_RASTER_RUNS
  c->stats.kernel_launches++;
  if (c->profile) {
    WRCU_CUDA(c, cudaEventRecord(c->p1, c->launch_stream));
    c->profile_valid = true;
  }
  WRCU_CUDA(c, cudaGetLastError());
  return WRCU_OK;
}


// ---- one set-up launch for every queued batch ---------------------------------------------------------
struct __align__(16) SetupJob {
  SetupArgs a;
  int kind;
  uint32_t features;
  int first_block;   // of this job in the launch
  int pad;
};
#ifndef WRCU_HOSTEMU
__global__ void __launch_bounds__(128) wr_setup_multi(const SetupJob* jobs, const int* block_job, BatchInfo* reset, int n_reset,
                                                      int* reset_ctr) {
  __shared__ SetupJob sj;
  if (blockIdx.x == 0) {  // re-arm the records the NEXT submission will use (the other half of the ring)
    for (int i = threadIdx.x; i < n_reset; i += blockDim.x) wr_reset_batch_info(reset + i);
    if (threadIdx.x < 2) reset_ctr[threadIdx.x] = 0;
  }
  const int j = __ldg(block_job + blockIdx.x);
  {
    const uint4* src = (const uint4*)(jobs + j);
    uint4* dst = (uint4*)&sj;
    for (int i = threadIdx.x; i < (int)(sizeof(SetupJob) / 16); i += blockDim.x) dst[i] = __ldg(src + i);
  }
  __syncthreads();
  const SetupArgs& a = sj.a;
  const int idx = ((int)blockIdx.x - sj.first_block) * (int)blockDim.x + (int)threadIdx.x;
  switch (sj.kind) {
    case WRCU_KIND_QUAD_TEXTURED: wr_setup_quad_textured_block(a, idx); break;
    case WRCU_KIND_QUAD_MASK: wr_setup_quad_mask_block(a, idx); break;
    case WRCU_KIND_BRUSH_SOLID: wr_setup_brush_solid_block(a, idx); break;
    case WRCU_KIND_BRUSH_IMAGE: wr_setup_brush_image_block(a, idx); break;
    case WRCU_KIND_BRUSH_LINEAR_GRADIENT: wr_setup_brush_linear_gradient_block(a, idx); break;
    case WRCU_KIND_BRUSH_BLEND: wr_setup_brush_blend_block(a, idx); break;
    case WRCU_KIND_BRUSH_MIX_BLEND: wr_setup_brush_mix_blend_block(a, idx); break;
    case WRCU_KIND_BRUSH_OPACITY: wr_setup_brush_opacity_block(a, idx); break;
    case WRCU_KIND_TEXT_RUN: wr_setup_text_run_block(a, idx); break;
    case WRCU_KIND_CLIP_RECTANGLE: wr_setup_clip_rectangle_block(a, idx); break;
    case WRCU_KIND_CLIP_BOX_SHADOW: wr_setup_clip_box_shadow_block(a, idx); break;
    case WRCU_KIND_COMPOSITE:
      if (sj.features & WRCU_FEAT_YUV) wr_setup_composite_yuv_block(a, idx);
      else wr_setup_composite_block(a, idx);
      break;
    case WRCU_KIND_CLEAR: wr_setup_clear_block(a, idx); break;
    case WRCU_KIND_BLUR: wr_setup_blur_block(a, idx); break;
    case WRCU_KIND_SCALE: wr_setup_scale_block(a, idx); break;
    case WRCU_KIND_FAST_LINEAR_GRADIENT: case WRCU_KIND_LINEAR_GRADIENT: case WRCU_KIND_RADIAL_GRADIENT:
    case WRCU_KIND_CONIC_GRADIENT: wr_setup_cs_gradient_block(a, idx); break;
    case WRCU_KIND_LINE_DECORATION: wr_setup_line_decoration_block(a, idx); break;
    case WRCU_KIND_BORDER_SOLID: case WRCU_KIND_BORDER_SEGMENT: wr_setup_border_block(a, idx); break;
    case WRCU_KIND_QUAD_RADIAL_GRADIENT: case WRCU_KIND_QUAD_CONIC_GRADIENT: wr_setup_quad_gradient_block(a, idx); break;
    case WRCU_KIND_BRUSH_YUV_IMAGE: wr_setup_brush_yuv_image_block(a, idx); break;
    case WRCU_KIND_SPLIT_COMPOSITE: wr_setup_split_composite_block(a, idx); break;
    default: break;
  }
}
#else
static void setup_host(int kind, uint32_t features, const SetupArgs& a) {
  switch (kind) {
    case WRCU_KIND_QUAD_TEXTURED: wr_setup_quad_textured(a); break;
    case WRCU_KIND_QUAD_MASK: wr_setup_quad_mask(a); break;
    case WRCU_KIND_BRUSH_SOLID: wr_setup_brush_solid(a); break;
    case WRCU_KIND_BRUSH_IMAGE: wr_setup_brush_image(a); break;
    case WRCU_KIND_BRUSH_LINEAR_GRADIENT: wr_setup_brush_linear_gradient(a); break;
    case WRCU_KIND_BRUSH_BLEND: wr_setup_brush_blend(a); break;
    case WRCU_KIND_BRUSH_MIX_BLEND: wr_setup_brush_mix_blend(a); break;
    case WRCU_KIND_BRUSH_OPACITY: wr_setup_brush_opacity(a); break;
    case WRCU_KIND_TEXT_RUN: wr_setup_text_run(a); break;
    case WRCU_KIND_CLIP_RECTANGLE: wr_setup_clip_rectangle(a); break;
    case WRCU_KIND_CLIP_BOX_SHADOW: wr_setup_clip_box_shadow(a); break;
    case WRCU_KIND_COMPOSITE:
      if (features & WRCU_FEAT_YUV) wr_setup_composite_yuv(a);
      else wr_setup_composite(a);
      break;
    case WRCU_KIND_CLEAR: wr_setup_clear(a); break;
    case WRCU_KIND_BLUR: wr_setup_blur(a); break;
    case WRCU_KIND_SCALE: wr_setup_scale(a); break;
    case WRCU_KIND_FAST_LINEAR_GRADIENT: case WRCU_KIND_LINEAR_GRADIENT: case WRCU_KIND_RADIAL_GRADIENT:
    case WRCU_KIND_CONIC_GRADIENT: wr_setup_cs_gradient(a); break;
    case WRCU_KIND_LINE_DECORATION: wr_setup_line_decoration(a); break;
    case WRCU_KIND_BORDER_SOLID: case WRCU_KIND_BORDER_SEGMENT: wr_setup_border(a); break;
    case WRCU_KIND_QUAD_RADIAL_GRADIENT: case WRCU_KIND_QUAD_CONIC_GRADIENT: wr_setup_quad_gradient(a); break;
    case WRCU_KIND_BRUSH_YUV_IMAGE: wr_setup_brush_yuv_image(a); break;
    case WRCU_KIND_SPLIT_COMPOSITE: wr_setup_split_composite(a); break;
    default: break;
  }
}
#endif

static int launch_clear(wrcu_ctx* c, const PendingOp& op);
static int launch_raster(wrcu_ctx* c, PendingOp& op);


#ifndef WRCU_HOSTEMU
// Render targets of one submission are mostly independent (picture-cache tiles never read each other,
// frame_builder.rs:995-1057; SURVEY.md §8e): their clears and raster launches go to a few side streams — one
// stream per target, round robin — so the small kernels of different tiles overlap instead of queueing behind
// one another (a page's tile pass is ~150 launches of 10-30 us each, nearly all latency).  Ordering that does
// matter is kept with events: an op waits for the latest earlier op on ANOTHER stream that wrote something it
// reads or writes, or read something it writes (colour target, depth target, sampled textures, clip mask).
// The side streams fork after the set-up launch and join before flush_pending returns, so everything outside
// the submission still sees one stream.
struct OpUse { const uint8_t* w[2]; int nw; const uint8_t* r[4]; int nr; };
static bool uses_conflict(const PendingOp& a, const OpUse& ua, const PendingOp& b, const OpUse& ub) {
  // a earlier, b later: RAW / WAW (a writes what b touches), WAR (a reads what b writes)
  for (int i = 0; i < ua.nw; i++) {
    for (int j = 0; j < ub.nw; j++) if (ua.w[i] == ub.w[j]) return true;
    for (int j = 0; j < ub.nr; j++) if (ua.w[i] == ub.r[j]) return true;
    for (const uint8_t* p : b.tex_reads) if (ua.w[i] == p) return true;
  }
  for (int j = 0; j < ub.nw; j++) {
    for (int i = 0; i < ua.nr; i++) if (ua.r[i] == ub.w[j]) return true;
    for (const uint8_t* p : a.tex_reads) if (p == ub.w[j]) return true;
  }
  return false;
}
static int ensure_side_streams(wrcu_ctx* c) {
  const int NS = c->n_streams;
  if (c->side.empty()) {
    c->side.resize((size_t)NS);
    for (int i = 0; i < NS; i++) WRCU_CUDA(c, cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking));
    WRCU_CUDA(c, cudaEventCreateWithFlags(&c->fork_ev, cudaEventDisableTiming));
    WRCU_CUDA(c, cudaEventCreateWithFlags(&c->fork0_ev, cudaEventDisableTiming));
    c->join_ev.resize((size_t)NS);
    for (int i = 0; i < NS; i++) WRCU_CUDA(c, cudaEventCreateWithFlags(&c->join_ev[i], cudaEventDisableTiming));
  }
  return WRCU_OK;
}
// Two fork points: `fork0_ev` was recorded before the submission's H2D copy and set-up launch — a stream that
// starts with clears (they read nothing the set-up writes) waits only for that and overlaps them — and
// `fork_ev` after the set-up launch, which every raster launch is behind.
static int flush_multi_stream(wrcu_ctx* c, std::vector<PendingOp>& q) {
  const int NS = c->n_streams;
  const size_t n = q.size();
  while (c->op_events.size() < n) {
    cudaEvent_t e;
    WRCU_CUDA(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->op_events.push_back(e);
  }
  std::vector<OpUse> use(n);
  std::vector<int> strm(n);
  std::vector<const uint8_t*> targets;
  for (size_t i = 0; i < n; i++) {
    const PendingOp& op = q[i];
    OpUse u;
    memset(&u, 0, sizeof u);
    const uint8_t* tgt = nullptr;
    if (op.type == 0) {
      if (op.c_ptr) u.w[u.nw++] = op.c_ptr;
      if (op.d_ptr) u.w[u.nw++] = op.d_ptr;
      tgt = op.c_ptr ? op.c_ptr : op.d_ptr;
    } else {
      u.w[u.nw++] = op.ra.tgt.color;
      if (op.ra.tgt.depth) u.w[u.nw++] = (const uint8_t*)op.ra.tgt.depth;
      const uint8_t* rs[4] = {op.sa.color0.ptr, op.sa.color1.ptr, op.sa.color2.ptr, op.sa.clip_mask.ptr};
      for (int k = 0; k < 4; k++) if (rs[k]) u.r[u.nr++] = rs[k];
      tgt = op.ra.tgt.color;
    }
    use[i] = u;
    size_t t = 0;
    while (t < targets.size() && targets[t] != tgt) t++;
    if (t == targets.size()) targets.push_back(tgt);
    strm[i] = (int)(t % (size_t)NS);
  }
  c->side_reduce = targets.size() >= 4;  // enough independent targets in flight to fill the chip between them
  // fork
  WRCU_CUDA(c, cudaEventRecord(c->fork_ev, c->stream));
  std::vector<char> used((size_t)NS, 0), need_ev(n, 0), behind_setup((size_t)NS, 0);
  std::vector<std::vector<int>> deps(n);
  for (size_t i = 0; i < n; i++) {
    // latest conflicting earlier op on each other stream
    std::vector<int> last((size_t)NS, -1);
    for (size_t j = 0; j < i; j++) {
      if (strm[j] == strm[i]) continue;
      if (uses_conflict(q[j], use[j], q[i], use[i])) last[(size_t)strm[j]] = (int)j;
    }
    for (int sidx = 0; sidx < NS; sidx++)
      if (last[(size_t)sidx] >= 0) { deps[i].push_back(last[(size_t)sidx]); need_ev[(size_t)last[(size_t)sidx]] = 1; }
  }
  for (size_t i = 0; i < n; i++) {
    PendingOp& op = q[i];
    cudaStream_t st = c->side[(size_t)strm[i]];
    c->plain_next = false;
    if (op.type == 0 && c->early_clear) {
      if (!used[(size_t)strm[i]]) WRCU_CUDA(c, cudaStreamWaitEvent(st, c->fork0_ev, 0));
    } else if (!behind_setup[(size_t)strm[i]]) {
      behind_setup[(size_t)strm[i]] = 1;
      WRCU_CUDA(c, cudaStreamWaitEvent(st, c->fork_ev, 0));
      c->plain_next = true;
    }
    used[(size_t)strm[i]] = 1;
    for (int j : deps[i]) {
      WRCU_CUDA(c, cudaStreamWaitEvent(st, c->op_events[(size_t)j], 0));
      c->plain_next = true;
    }
    c->launch_stream = st;
    if (op.type == 1) op.ra.pdl_early = c->pdl ? 1 : 0;  // the set-up launch finished before the fork event
    int rc = op.type == 0 ? launch_clear(c, op) : launch_raster(c, op);
    if (rc != WRCU_OK) { c->launch_stream = c->stream; c->side_reduce = false; return rc; }
    if (need_ev[i]) WRCU_CUDA(c, cudaEventRecord(c->op_events[i], st));
  }
  c->launch_stream = c->stream;
  c->side_reduce = false;
  c->plain_next = false;
  // join
  for (int sidx = 0; sidx < NS; sidx++) {
    if (!used[(size_t)sidx]) continue;
    WRCU_CUDA(c, cudaEventRecord(c->join_ev[(size_t)sidx], c->side[(size_t)sidx]));
    WRCU_CUDA(c, cudaStreamWaitEvent(c->stream, c->join_ev[(size_t)sidx], 0));
  }
  return WRCU_OK;
}
#endif

static int flush_pending(wrcu_ctx* c) {
  if (c->in_flush) return WRCU_OK;
  std::vector<PendingOp>& q = pending(c);
  if (q.empty() && c->dirty_hi <= c->dirty_lo) return WRCU_OK;
  cudaSetDevice(c->device);
  c->in_flush = true;
  struct Guard { wrcu_ctx* c; std::vector<PendingOp>& q; ~Guard() { q.clear(); c->pend_instances = 0; c->in_flush = false; } } guard{c, q};
  size_t total_n = 0, bin_total = 0;
  int nb = 0, total_blocks = 0;
  for (const PendingOp& op : q)
    if (op.type == 1) { total_n += (size_t)op.n; bin_total += op.bin_need; nb++; total_blocks += op.sblocks; }
  BatchInfo* infos = (BatchInfo*)c->batch_info + (size_t)c->flush_parity * wrcu_ctx::QMAX;
  BatchInfo* infos_next = (BatchInfo*)c->batch_info + (size_t)(c->flush_parity ^ 1) * wrcu_ctx::QMAX;
  int* ctr = c->pool_ctr + c->flush_parity * 2;
  int* ctr_next = c->pool_ctr + (c->flush_parity ^ 1) * 2;
  size_t jobs_off = 0, map_off = 0;
  if (nb) {
    int rc;
    if ((rc = ensure_cmd_capacity(c, total_n)) != WRCU_OK) return rc;
    if (bin_total > c->bin_cap_words) {
      WRCU_CUDA(c, cudaStreamSynchronize(c->stream));
      if (c->bin_mask) cudaFree(c->bin_mask);
      c->bin_mask = nullptr;
      c->bin_cap_words = 0;
      WRCU_CUDA(c, cudaMalloc((void**)&c->bin_mask, bin_total * 4 * 2));
      c->bin_cap_words = bin_total * 2;
    }
    // the job table lives in the arena too; reserving it may still move the arena (pointers are resolved below)
    if ((rc = arena_reserve(c, (size_t)nb * sizeof(SetupJob), &jobs_off)) != WRCU_OK) return rc;
    if ((rc = arena_reserve(c, (size_t)total_blocks * sizeof(int), &map_off)) != WRCU_OK) return rc;
    Arena* a = &c->arena[c->cur_arena];
    SetupJob* jobs = (SetupJob*)(a->host + jobs_off);
    int* block_job = (int*)(a->host + map_off);
    size_t off = 0, boff = 0;
    int bi = 0, blk = 0;
    for (PendingOp& op : q) {
      if (op.type != 1) continue;
      SetupArgs& sa = op.sa;
      RasterArgs& ra = op.ra;
      sa.tabs = c->tables;
      sa.instances = a->dev + op.inst_off;
      sa.tex_list = op.views_off != (size_t)-1 ? (const TexView*)(a->dev + op.views_off) : nullptr;
      sa.hot = (CmdHot*)c->cmd_hot + off;
      sa.cold = (CmdCold*)c->cmd_cold + off;
      sa.info = infos + bi;
      sa.info_next = nullptr;
      sa.pool_ctr = ctr;
      sa.row_tab = c->row_tab;
      sa.row_cap = c->row_cap;
      if (op.bin_need) {
        const size_t words = (size_t)sa.bin_words, tiles = (op.bin_need - 2 * (size_t)sa.any_words - 1) / words - 1;
        sa.tile_mask = c->bin_mask + boff;
        sa.wide_mask = sa.tile_mask + tiles * words;
        sa.tile_any = sa.wide_mask + words;
        boff += op.bin_need;
      }
      ra.hot = sa.hot;
      ra.cold = sa.cold;
      ra.info = sa.info;
      ra.tile_mask = sa.tile_mask;
      ra.wide_mask = sa.wide_mask;
      ra.tile_any = sa.tile_any;
      ra.tile_ord = sa.tile_any ? sa.tile_any + sa.any_words + 1 : nullptr;
      ra.row_tab = c->row_tab;
      ra.gbuf_f = c->tables.gpu_buffer_f;
      ra.n_gbuf_f = c->tables.n_gpu_buffer_f;
      ra.gpu_cache = c->tables.gpu_cache;
      ra.n_gpu_cache = c->tables.n_gpu_cache;
      memset(&jobs[bi], 0, sizeof(SetupJob));
      jobs[bi].a = sa;
      jobs[bi].kind = op.kind;
      jobs[bi].features = op.features;
      jobs[bi].first_block = blk;
      for (int k = 0; k < op.sblocks; k++) block_job[blk + k] = bi;
      blk += op.sblocks;
      off += (size_t)op.n;
      bi++;
    }
    mark_dirty(c, jobs_off, jobs_off + (size_t)nb * sizeof(SetupJob));
    mark_dirty(c, map_off, map_off + (size_t)total_blocks * sizeof(int));
    c->stats.h2d_bytes += (size_t)nb * sizeof(SetupJob) + (size_t)total_blocks * sizeof(int);
  }
#ifndef WRCU_HOSTEMU
  // several launches, or a clear ahead of a draw: side streams (the clear overlaps the copy and the set-up launch)
  const bool multi = c->n_streams > 1 && (q.size() > 2 || (c->early_clear && q.size() == 2 && q[0].type == 0 && q[1].type == 1));
  if (multi) {
    int rce = ensure_side_streams(c);
    if (rce != WRCU_OK) return rce;
    WRCU_CUDA(c, cudaEventRecord(c->fork0_ev, c->stream));
  }
#endif
  if (c->dirty_hi > c->dirty_lo) {
    Arena* a = &c->arena[c->cur_arena];
    WRCU_CUDA(c, cudaMemcpyAsync(a->dev + c->dirty_lo, a->host + c->dirty_lo, c->dirty_hi - c->dirty_lo, cudaMemcpyHostToDevice,
                                 c->stream));
    c->dirty_lo = c->dirty_hi = 0;
  }
  if (nb) {
    Arena* a = &c->arena[c->cur_arena];
    if (bin_total) WRCU_CUDA(c, cudaMemsetAsync(c->bin_mask, 0, bin_total * 4, c->stream));
#ifndef WRCU_HOSTEMU
    wr_setup_multi<<<total_blocks, 128, 0, c->stream>>>((const SetupJob*)(a->dev + jobs_off), (const int*)(a->dev + map_off), infos_next,
                                                        wrcu_ctx::QMAX, ctr_next);
    c->stats.kernel_launches++;
    WRCU_CUDA(c, cudaGetLastError());
#else
    for (int i = 0; i < wrcu_ctx::QMAX; i++) wr_reset_batch_info(infos_next + i);
    ctr_next[0] = ctr_next[1] = 0;
    for (PendingOp& op : q)
      if (op.type == 1) setup_host(op.kind, op.features, op.sa);
#endif
  }
  c->launch_stream = c->stream;
#ifndef WRCU_HOSTEMU
  if (multi) {
    int rcs = flush_multi_stream(c, q);
    if (rcs != WRCU_OK) return rcs;
    if (nb) c->flush_parity ^= 1;
    return WRCU_OK;
  }
#endif
  bool after_setup = nb > 0;  // the first raster launch follows the set-up launch: it must wait before reading commands
  for (PendingOp& op : q) {
    if (op.type == 1) {
      op.ra.pdl_early = (c->pdl && !after_setup) ? 1 : 0;
      after_setup = false;
    }
    int rc = op.type == 0 ? launch_clear(c, op) : launch_raster(c, op);
    if (rc != WRCU_OK) return rc;
  }
  if (nb) c->flush_parity ^= 1;
  return WRCU_OK;
}

extern "C" int wrcu_program_from_name(const char* key, int* kind, uint32_t* features) {
  if (!key || !kind || !features) return WRCU_ERR_INVALID;
  static const struct { const char* name; int kind; } names[] = {
      {"ps_quad_textured", WRCU_KIND_QUAD_TEXTURED}, {"ps_quad_mask", WRCU_KIND_QUAD_MASK},
      {"brush_solid", WRCU_KIND_BRUSH_SOLID}, {"brush_image", WRCU_KIND_BRUSH_IMAGE},
      {"brush_linear_gradient", WRCU_KIND_BRUSH_LINEAR_GRADIENT}, {"brush_blend", WRCU_KIND_BRUSH_BLEND},
      {"brush_mix_blend", WRCU_KIND_BRUSH_MIX_BLEND}, {"brush_opacity", WRCU_KIND_BRUSH_OPACITY},
      {"ps_text_run", WRCU_KIND_TEXT_RUN}, {"cs_clip_rectangle", WRCU_KIND_CLIP_RECTANGLE},
      {"cs_clip_box_shadow", WRCU_KIND_CLIP_BOX_SHADOW}, {"composite", WRCU_KIND_COMPOSITE}, {"brush_yuv_image", WRCU_KIND_BRUSH_YUV_IMAGE},
      {"ps_split_composite", WRCU_KIND_SPLIT_COMPOSITE},
      {"ps_clear", WRCU_KIND_CLEAR}, {"cs_blur", WRCU_KIND_BLUR}, {"cs_scale", WRCU_KIND_SCALE},
      {"cs_fast_linear_gradient", WRCU_KIND_FAST_LINEAR_GRADIENT}, {"cs_linear_gradient", WRCU_KIND_LINEAR_GRADIENT},
      {"cs_radial_gradient", WRCU_KIND_RADIAL_GRADIENT}, {"cs_conic_gradient", WRCU_KIND_CONIC_GRADIENT},
      {"cs_line_decoration", WRCU_KIND_LINE_DECORATION}, {"cs_border_solid", WRCU_KIND_BORDER_SOLID},
      {"cs_border_segment", WRCU_KIND_BORDER_SEGMENT}, {"ps_quad_radial_gradient", WRCU_KIND_QUAD_RADIAL_GRADIENT},
      {"ps_quad_conic_gradient", WRCU_KIND_QUAD_CONIC_GRADIENT}};
  static const struct { const char* name; uint32_t bit; } feats[] = {
      {"ALPHA_PASS", WRCU_FEAT_ALPHA_PASS}, {"FAST_PATH", WRCU_FEAT_FAST_PATH},
      {"ANTIALIASING", WRCU_FEAT_ANTIALIASING}, {"REPETITION", WRCU_FEAT_REPETITION},
      {"DUAL_SOURCE_BLENDING", WRCU_FEAT_DUAL_SOURCE_BLENDING}, {"ADVANCED_BLEND", WRCU_FEAT_ADVANCED_BLEND},
      {"GLYPH_TRANSFORM", WRCU_FEAT_GLYPH_TRANSFORM}, {"TEXTURE_2D", WRCU_FEAT_TEXTURE_2D},
      {"ALPHA_TARGET", WRCU_FEAT_ALPHA_TARGET}, {"COLOR_TARGET", WRCU_FEAT_COLOR_TARGET},
      {"YUV", WRCU_FEAT_YUV}};
  const char* sp = strchr(key, ' ');
  size_t nlen = sp ? (size_t)(sp - key) : strlen(key);
  *kind = 0;
  for (auto& e : names)
    if (strlen(e.name) == nlen && !strncmp(e.name, key, nlen)) *kind = e.kind;
  if (!*kind) return WRCU_ERR_UNSUPPORTED;
  *features = 0;
  const char* p = sp ? sp + 1 : nullptr;
  while (p && *p) {
    const char* comma = strchr(p, ',');
    size_t flen = comma ? (size_t)(comma - p) : strlen(p);
    bool found = false;
    for (auto& f : feats)
      if (strlen(f.name) == flen && !strncmp(f.name, p, flen)) {
        *features |= f.bit;
        found = true;
      }
    if (!found) return WRCU_ERR_UNSUPPORTED;  // TEXTURE_RECT, TEXTURE_EXTERNAL, DEBUG_OVERDRAW, ...
    p = comma ? comma + 1 : nullptr;
  }
  return WRCU_OK;
}

// ---- stats / timing ---------------------------------------------------------------------
extern "C" int wrcu_get_stats(wrcu_ctx* c, wrcu_stats* out) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  *out = c->stats;
  return WRCU_OK;
}
extern "C" int wrcu_reset_stats(wrcu_ctx* c) {
  memset(&c->stats, 0, sizeof c->stats);
  return WRCU_OK;
}
extern "C" int wrcu_profile_enable(wrcu_ctx* c, int on) {
  c->profile = on != 0;
  c->profile_valid = false;
  return WRCU_OK;
}
extern "C" int wrcu_last_raster_ms(wrcu_ctx* c, float* ms) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  if (!ms || !c->profile_valid) return wrcu_fail(c, WRCU_ERR_INVALID, "last_raster_ms: no profiled draw");
  WRCU_CUDA(c, cudaEventSynchronize(c->p1));
  WRCU_CUDA(c, cudaEventElapsedTime(ms, c->p0, c->p1));
  return WRCU_OK;
}
extern "C" int wrcu_timer_begin(wrcu_ctx* c) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WRCU_CUDA(c, cudaEventRecord(c->t0, c->stream));
  return WRCU_OK;
}
extern "C" int wrcu_timer_end(wrcu_ctx* c, float* ms) {
  { int rcf_ = flush_pending(c); if (rcf_ != WRCU_OK) return rcf_; }
  WRCU_CUDA(c, cudaEventRecord(c->t1, c->stream));
  WRCU_CUDA(c, cudaEventSynchronize(c->t1));
  WRCU_CUDA(c, cudaEventElapsedTime(ms, c->t0, c->t1));
  return WRCU_OK;
}
