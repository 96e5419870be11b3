/* wrcu.h — C ABI of the B200-native WebRender frame-draw backend.
 *
 * This is the drop-in boundary for ONE path of servo/webrender: the render
 * thread's `Renderer::draw_frame` (webrender/src/renderer/mod.rs:4525) and the
 * device calls it makes — `draw_instanced_batch` (mod.rs:2022), target binds,
 * clears, clip-mask batches and the final tile composite.  In the reference
 * those calls go through `Device` to the `gleam::gl::Gl` trait object
 * (renderer/init.rs:292-297); with the software rasteriser the trait is
 * implemented by 99 `extern "C"` symbols (swgl/src/swgl_fns.rs:23-320 →
 * swgl/src/gl.cc:1080-2851).  This header is the "thin FFI" version of that
 * seam (SURVEY.md §8b option 2): every entry point names the reference call
 * sequence it replaces.  Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions
 *  - Every function returns WRCU_OK (0) or a negative wrcu_status; nothing
 *    throws or aborts across the ABI.  Like GL (gl.cc:1126-1134) the context
 *    also keeps a sticky error readable with wrcu_get_error().
 *  - The host owns every array it passes in; the backend copies what it needs
 *    before the call returns (the reference copies at glBufferData time,
 *    device/gl.rs:3552-3600).
 *  - Work is queued on a CUDA stream; wrcu_read_pixels / wrcu_finish
 *    synchronise (the SWGL equivalents are synchronous, gl.cc:2802).
 *    wrcu_clear and wrcu_draw_batch / wrcu_draw_composite_tiles are further
 *    queued inside the library and submitted together — one host-to-device
 *    copy and one set-up launch for every queued batch — by the next call of
 *    any other kind (wrcu_frame_end at the latest), so their execution order
 *    relative to every other call is exactly the call order.  Asynchronous
 *    errors of a draw (an instance the backend cannot rasterise) surface at
 *    the next synchronising call, as GL errors do.
 *  - One context per host thread, like `MakeCurrent` (gl.cc:2808).
 *  - Colour targets are "RGBA8" with B,G,R,A byte order in memory exactly as
 *    SWGL stores them (swgl/src/texture.h:85-90); alpha targets are R8.
 */
#ifndef WRCU_H
#define WRCU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WRCU_ABI_VERSION 1

typedef struct wrcu_ctx wrcu_ctx;
typedef uint32_t wrcu_tex; /* 0 = none; like a GLuint texture name */

typedef enum wrcu_status {
  WRCU_OK = 0,
  WRCU_ERR_INVALID = -1,      /* bad argument / unknown handle            */
  WRCU_ERR_OOM = -2,          /* GL_OUT_OF_MEMORY (gl.cc:1134)            */
  WRCU_ERR_CUDA = -3,         /* a CUDA runtime call failed               */
  WRCU_ERR_UNSUPPORTED = -4,  /* valid in the reference, not built here   */
  WRCU_ERR_NO_DEVICE = -5     /* no usable CUDA device (never falls back) */
} wrcu_status;

/* Texture formats (gl.cc:216-260 bytes_for_internal_format). */
typedef enum wrcu_format {
  WRCU_FMT_RGBA8 = 1,   /* 4 B/px, BGRA in memory                         */
  WRCU_FMT_R8 = 2,      /* 1 B/px                                         */
  WRCU_FMT_RGBAF32 = 3, /* 16 B/texel (data textures, GPU cache)          */
  WRCU_FMT_RGBAI32 = 4, /* 16 B/texel                                     */
  WRCU_FMT_DEPTH24 = 5, /* 4 B/px, 24-bit depth (rasterize.h:37)          */
  WRCU_FMT_RG8 = 6,     /* 2 B/px, sample-only: the CbCr plane of NV12 video
                           surfaces (gl.cc:247, TextureFormat::RG8)          */
  WRCU_FMT_R16 = 7,     /* 2 B/px, sample-only: a 10/12/16-bit video plane
                           (gl.cc:257, TextureFormat::R16)                   */
  WRCU_FMT_RG16 = 8     /* 4 B/px, sample-only: the CbCr plane of 10/12/16-bit
                           NV12 and P010 surfaces (gl.cc:259, TextureFormat::RG16) */
} wrcu_format;

typedef enum wrcu_filter { WRCU_NEAREST = 0, WRCU_LINEAR = 1 } wrcu_filter;

/* Batch kinds = the reference's shader programs (SURVEY.md §2.3, Appendix C;
 * BatchKind in webrender/src/batch.rs:60-86, shader table renderer/shade.rs). */
typedef enum wrcu_kind {
  WRCU_KIND_QUAD_TEXTURED = 1,         /* ps_quad_textured                 */
  WRCU_KIND_QUAD_MASK = 2,             /* ps_quad_mask [FAST_PATH]         */
  WRCU_KIND_BRUSH_SOLID = 3,           /* brush_solid                      */
  WRCU_KIND_BRUSH_IMAGE = 4,           /* brush_image                      */
  WRCU_KIND_BRUSH_LINEAR_GRADIENT = 5, /* brush_linear_gradient            */
  WRCU_KIND_BRUSH_BLEND = 6,           /* brush_blend                      */
  WRCU_KIND_BRUSH_MIX_BLEND = 7,       /* brush_mix_blend                  */
  WRCU_KIND_BRUSH_OPACITY = 8,         /* brush_opacity                    */
  WRCU_KIND_TEXT_RUN = 9,              /* ps_text_run                      */
  WRCU_KIND_CLIP_RECTANGLE = 10,       /* cs_clip_rectangle [FAST_PATH]    */
  WRCU_KIND_CLIP_BOX_SHADOW = 11,      /* cs_clip_box_shadow               */
  WRCU_KIND_COMPOSITE = 12,            /* composite [FAST_PATH | YUV]      */
  WRCU_KIND_CLEAR = 13,                /* ps_clear                         */
  WRCU_KIND_BLUR = 14,                 /* cs_blur (SURVEY §8f rank 1)      */
  WRCU_KIND_SCALE = 15,                /* cs_scale                         */
  /* texture-cache-target render tasks (SURVEY §8f rank 2; renderer/mod.rs:3931-4200) */
  WRCU_KIND_FAST_LINEAR_GRADIENT = 16, /* cs_fast_linear_gradient          */
  WRCU_KIND_LINEAR_GRADIENT = 17,      /* cs_linear_gradient               */
  WRCU_KIND_RADIAL_GRADIENT = 18,      /* cs_radial_gradient               */
  WRCU_KIND_CONIC_GRADIENT = 19,       /* cs_conic_gradient                */
  WRCU_KIND_LINE_DECORATION = 20,      /* cs_line_decoration               */
  WRCU_KIND_BORDER_SOLID = 21,         /* cs_border_solid                  */
  WRCU_KIND_BORDER_SEGMENT = 22,       /* cs_border_segment                */
  WRCU_KIND_QUAD_RADIAL_GRADIENT = 23, /* ps_quad_radial_gradient          */
  WRCU_KIND_QUAD_CONIC_GRADIENT = 24,  /* ps_quad_conic_gradient           */
  WRCU_KIND_BRUSH_YUV_IMAGE = 25,      /* brush_yuv_image [ALPHA_PASS] YUV: BrushBatchKind::YuvImage
                                          (batch.rs:60-86), planes in color[0..2]  */
  WRCU_KIND_SPLIT_COMPOSITE = 26       /* ps_split_composite: BatchKind::SplitComposite (batch.rs:74), instances =
                                          SplitCompositeInstance (gpu_types.rs:531-552), surface in color[0] */
} wrcu_kind;

/* Shader feature bits (webrender_build/src/shader_features.rs:64-247). */
enum {
  WRCU_FEAT_ALPHA_PASS = 1u << 0,
  WRCU_FEAT_FAST_PATH = 1u << 1,
  WRCU_FEAT_ANTIALIASING = 1u << 2,
  WRCU_FEAT_REPETITION = 1u << 3,
  WRCU_FEAT_DUAL_SOURCE_BLENDING = 1u << 4,
  WRCU_FEAT_ADVANCED_BLEND = 1u << 5,
  WRCU_FEAT_GLYPH_TRANSFORM = 1u << 6,
  WRCU_FEAT_TEXTURE_2D = 1u << 7,
  WRCU_FEAT_ALPHA_TARGET = 1u << 8, /* cs_blur into an R8 target    */
  WRCU_FEAT_COLOR_TARGET = 1u << 9, /* cs_blur into an RGBA8 target */
  WRCU_FEAT_YUV = 1u << 10          /* composite: YUV video surfaces (composite.glsl:14-33),
                                       8-bit PLANAR / NV12 / INTERLEAVED planes;
                                       10/12/16-bit PLANAR (3 x R16), NV12 and P010
                                       (R16 + RG16)                                */
};

/* Blend keys: exactly the set the reference's blend stage implements
 * (FOR_EACH_BLEND_KEY, swgl/src/gl.cc:617-649), i.e. what the Device blend
 * setters reduce to (device/gl.rs:3901-4017 → gl.cc:1240-1335).  Blending
 * disabled = WRCU_BLEND_NONE. */
typedef enum wrcu_blend {
  WRCU_BLEND_NONE = 0,              /* ONE, ZERO / blending off            */
  WRCU_BLEND_ALPHA = 1,             /* SRC_ALPHA,1-SRC_ALPHA,ONE,1-SRC_ALPHA */
  WRCU_BLEND_PREMULTIPLIED_ALPHA = 2,   /* ONE, 1-SRC_ALPHA                */
  WRCU_BLEND_SUBPIXEL_PASS0 = 3,        /* ZERO, 1-SRC_COLOR               */
  WRCU_BLEND_SUBPIXEL_PASS0_KEEP_A = 4, /* ZERO,1-SRC_COLOR,ZERO,ONE       */
  WRCU_BLEND_PREMULTIPLIED_DEST_OUT = 5, /* ZERO, 1-SRC_ALPHA              */
  WRCU_BLEND_MULTIPLY = 6,              /* ZERO, SRC_COLOR (clip masks)    */
  WRCU_BLEND_PLUS_LIGHTER = 7,          /* ONE, ONE                        */
  WRCU_BLEND_ADD_KEEP_ALPHA_OVER = 8,   /* ONE,ONE,ONE,1-SRC_ALPHA         */
  WRCU_BLEND_DST_ALPHA_ADD = 9,         /* 1-DST_ALPHA,ONE,ZERO,ONE        */
  WRCU_BLEND_CONSTANT_COLOR = 10,       /* CONSTANT_COLOR, 1-SRC_COLOR     */
  WRCU_BLEND_SUBPIXEL_DUAL_SOURCE = 11, /* ONE, 1-SRC1_COLOR               */
  WRCU_BLEND_MIN = 12,
  WRCU_BLEND_MAX = 13,
  /* KHR_blend_equation_advanced (MixBlendMode → device/gl.rs:3996-4017) */
  WRCU_BLEND_ADV_MULTIPLY = 14,
  WRCU_BLEND_ADV_SCREEN = 15,
  WRCU_BLEND_ADV_OVERLAY = 16,
  WRCU_BLEND_ADV_DARKEN = 17,
  WRCU_BLEND_ADV_LIGHTEN = 18,
  WRCU_BLEND_ADV_COLOR_DODGE = 19,
  WRCU_BLEND_ADV_COLOR_BURN = 20,
  WRCU_BLEND_ADV_HARD_LIGHT = 21,
  WRCU_BLEND_ADV_SOFT_LIGHT = 22,
  WRCU_BLEND_ADV_DIFFERENCE = 23,
  WRCU_BLEND_ADV_EXCLUSION = 24,
  WRCU_BLEND_ADV_HUE = 25,
  WRCU_BLEND_ADV_SATURATION = 26,
  WRCU_BLEND_ADV_COLOR = 27,
  WRCU_BLEND_ADV_LUMINOSITY = 28,
  WRCU_BLEND__COUNT
} wrcu_blend;

typedef enum wrcu_depth {
  WRCU_DEPTH_OFF = 0,          /* depth test disabled                      */
  WRCU_DEPTH_TEST = 1,         /* LEQUAL test, no write (alpha pass)       */
  WRCU_DEPTH_TEST_WRITE = 2    /* LEQUAL test + write (opaque pass)        */
} wrcu_depth;

/* Per-frame data tables = the 1024-texel-wide data textures the reference
 * uploads in bind_frame_data / prepare_gpu_cache (renderer/mod.rs:4418,
 * 1536; renderer/vertex.rs:984-1038).  Counts are in 16-byte texels ("vec4
 * blocks"); addresses inside instance data index these arrays linearly
 * (address -> (a % 1024, a / 1024) in the reference, res/gpu_cache.glsl:16). */
typedef struct wrcu_frame_tables {
  const float* prim_headers_f;   size_t prim_headers_f_texels;  /* 2/prim  */
  const int32_t* prim_headers_i; size_t prim_headers_i_texels;  /* 2/prim  */
  const float* transforms;       size_t transforms_texels;      /* 8/xform */
  const float* render_tasks;     size_t render_tasks_texels;    /* 2/task  */
  const float* gpu_cache;        size_t gpu_cache_texels;
  const float* gpu_buffer_f;     size_t gpu_buffer_f_texels;
  const int32_t* gpu_buffer_i;   size_t gpu_buffer_i_texels;
} wrcu_frame_tables;

/* State a draw depends on (SURVEY.md §8b last row): what the reference holds
 * in GL state — bound textures (renderer/mod.rs:369-386), blend, depth,
 * scissor — passed explicitly. */
typedef struct wrcu_draw_state {
  int32_t blend;        /* wrcu_blend                                      */
  int32_t depth;        /* wrcu_depth                                      */
  wrcu_tex color[3];    /* sColor0..2                                      */
  wrcu_tex clip_mask;   /* sClipMask (BatchTextures.clip_mask)             */
  int32_t scissor_enabled;
  int32_t scissor[4];   /* x, y, w, h — device pixels, GL SetScissor       */
  float blend_color[4]; /* glBlendColor, for WRCU_BLEND_CONSTANT_COLOR     */
} wrcu_draw_state;

/* ---- context ----------------------------------------------------------- */
/* CreateContext/MakeCurrent (gl.cc:2806-2818).  device_ordinal = CUDA device. */
int wrcu_ctx_create(int device_ordinal, wrcu_ctx** out);
void wrcu_ctx_destroy(wrcu_ctx* ctx);                 /* DestroyContext     */
int wrcu_get_error(wrcu_ctx* ctx);                    /* GetError, sticky   */
const char* wrcu_last_error_string(wrcu_ctx* ctx);
const char* wrcu_get_string(int what);                /* GetString: 0=renderer
        returns "Software WebRender" so the host keeps is_software behaviour
        (gl.cc:1214, device/gl.rs:1645) ; 1=backend description              */
int wrcu_abi_version(void);
int wrcu_finish(wrcu_ctx* ctx);                       /* Finish (gl.cc:2802) */

/* ---- textures / render targets ------------------------------------------ */
/* GenTextures + TexStorage2D (gl.cc:1755, 1863). */
int wrcu_texture_create(wrcu_ctx* ctx, int format, int width, int height,
                        wrcu_tex* out);
/* SetTextureParameter MAG/MIN filter (gl.cc:1838). */
int wrcu_texture_set_filter(wrcu_ctx* ctx, wrcu_tex tex, int filter);
/* TexSubImage2D (gl.cc:1794): rows are `src_stride` bytes apart. */
int wrcu_texture_upload(wrcu_ctx* ctx, wrcu_tex tex, int x, int y, int w, int h,
                        const void* data, size_t src_stride);
int wrcu_texture_destroy(wrcu_ctx* ctx, wrcu_tex tex);   /* DeleteTexture   */
/* ReadPixels (gl.cc:2562): synchronises. */
int wrcu_read_pixels(wrcu_ctx* ctx, wrcu_tex tex, int x, int y, int w, int h,
                     void* out, size_t dst_stride);

/* ---- update path (SURVEY.md §8f rank 3: the step before the draws) ---------- */
/* Batched texture-cache upload: update_texture_cache → upload_to_texture_cache
 * (renderer/mod.rs:1795-1990, renderer/upload.rs:67-330).  The reference packs
 * the frame's small updates into PBO-backed staging buffers and copies them into
 * place; here `staging` (host memory; page-locked memory from wrcu_host_alloc is
 * copied without an intermediate pass) crosses PCIe in ONE transfer and one
 * kernel scatters every rect into the texture.  Rect i reads `h` rows of
 * `w * bytes_per_pixel` bytes, `stride` bytes apart, starting `offset` bytes
 * into `staging`. */
typedef struct wrcu_upload_rect {
  int32_t x, y, w, h;   /* destination rect in the texture                  */
  uint64_t offset;      /* byte offset of the first row inside `staging`    */
  uint64_t stride;      /* byte distance between source rows                */
} wrcu_upload_rect;
int wrcu_texture_upload_batch(wrcu_ctx* ctx, wrcu_tex tex,
                              const wrcu_upload_rect* rects, size_t n_rects,
                              const void* staging, size_t staging_bytes);
/* Texture-to-texture copy of a rect at 1:1: the texture-cache copies of
 * update_texture_cache (renderer/mod.rs:1808-1850, ps_copy) and handle_blits
 * (renderer/mod.rs:2438-2470).  src_rect = x, y, w, h. */
int wrcu_texture_copy(wrcu_ctx* ctx, wrcu_tex src, wrcu_tex dst,
                      const int32_t src_rect[4], int dst_x, int dst_y);
/* GPU cache updates: GpuCacheUpdateList applied by GpuCacheTexture::update +
 * flush (renderer/gpu_cache.rs:218-380, res/gpu_cache_update.glsl; update list
 * gpu_cache.rs:296-345).  The cache persists on the device across frames as
 * `height` rows of 1024 16-byte blocks (grown keeping its contents; `clear`
 * zeroes it first).  Each Copy scatters block_count blocks from
 * blocks[block_index..] to row v, column u.  Once this has been called,
 * wrcu_frame_begin accepts tables->gpu_cache == NULL (with gpu_cache_texels 0)
 * and binds the persistent cache, as the reference binds its GPU cache texture. */
typedef struct wrcu_gpu_cache_copy {
  uint32_t block_index, block_count;
  uint16_t u, v;        /* GpuCacheAddress                                  */
} wrcu_gpu_cache_copy;
int wrcu_gpu_cache_update(wrcu_ctx* ctx, int height, int clear,
                          const wrcu_gpu_cache_copy* updates, size_t n_updates,
                          const float* blocks, size_t n_blocks);

/* ---- frame --------------------------------------------------------------- */
/* bind_frame_data + gpu_buffer textures + prepare_gpu_cache
 * (renderer/mod.rs:4418, 4551-4558, 1536). */
int wrcu_frame_begin(wrcu_ctx* ctx, const wrcu_frame_tables* tables);
int wrcu_frame_end(wrcu_ctx* ctx);   /* end_frame / gl.flush (mod.rs:4820) */

/* ---- target binding, clears ---------------------------------------------- */
/* bind_draw_target + uTransform + viewport (device/gl.rs:2130-2180,
 * renderer/mod.rs:4705-4712).  `projection` is the column-major 4x4 ortho
 * matrix the reference passes as uTransform; viewport is x,y,w,h.
 * depth = 0 → no depth attachment. */
int wrcu_target_bind(wrcu_ctx* ctx, wrcu_tex color, wrcu_tex depth,
                     const float projection[16], const int32_t viewport[4]);
/* clear_target (device/gl.rs:3779-3830 → gl.cc:2498 Clear).  rect NULL =
 * whole target; color NULL = leave colour; depth NULL = leave depth. */
int wrcu_clear(wrcu_ctx* ctx, const int32_t rect[4], const float color[4],
               const float* depth);

/* ---- draws ---------------------------------------------------------------- */
/* draw_instanced_batch (renderer/mod.rs:2022-2065) =
 *   bind_textures + update_vao_instances (glBufferData) +
 *   glDrawElementsInstanced(TRIANGLES, 6, u16, 0, n) (gl.cc:2702).
 * `instances` is the tightly packed #[repr(C)] instance array for `kind`
 * (webrender/src/gpu_types.rs; SURVEY.md Appendix B); `instance_stride` its
 * element size in bytes.  Instances are drawn in order. */
int wrcu_draw_batch(wrcu_ctx* ctx, int kind, uint32_t features,
                    const wrcu_draw_state* state, const void* instances,
                    size_t instance_stride, int n_instances);

/* draw_tile_list (renderer/mod.rs:3126-3334) in one submission.  The reference has to break its
 * CompositeInstance list into a GL draw whenever the tile texture changes (mod.rs:3289-3316): one
 * draw per picture-cache tile.  Here the texture of every instance travels with it — `textures[i]`
 * is sColor0 of instance i, `state->color[0]` is ignored — so a whole tile list with the same shader
 * parameters (`features`: TEXTURE_2D, optionally FAST_PATH) and blend state is two kernel launches.
 * Instances are drawn in order; results equal n wrcu_draw_batch(WRCU_KIND_COMPOSITE, ..) calls. */
int wrcu_draw_composite_tiles(wrcu_ctx* ctx, uint32_t features,
                              const wrcu_draw_state* state, const void* instances,
                              size_t instance_stride, int n_instances,
                              const wrcu_tex* textures);

/* Program-key lookup: maps the reference's program name string
 * "<shader>[ FEAT,FEAT]" (swgl/build.rs:13-31, gl.cc:1431) to kind+features.
 * Returns WRCU_ERR_UNSUPPORTED for programs outside the hot path. */
int wrcu_program_from_name(const char* key, int* kind, uint32_t* features);

/* ---- statistics ------------------------------------------------------------ */
typedef struct wrcu_stats {
  uint64_t kernel_launches;   /* kernels of THIS library launched so far   */
  uint64_t draw_calls;        /* wrcu_draw_batch calls                      */
  uint64_t instances;         /* instances submitted                        */
  uint64_t h2d_bytes;         /* host→device bytes copied                   */
  uint64_t d2h_bytes;         /* device→host bytes copied                   */
} wrcu_stats;
int wrcu_get_stats(wrcu_ctx* ctx, wrcu_stats* out);
int wrcu_reset_stats(wrcu_ctx* ctx);

/* Device-side timing of the draws issued between begin/end, CUDA events on
 * the context's stream (the reference's GpuTimer, device/query_gl.rs:20-31). */
int wrcu_timer_begin(wrcu_ctx* ctx);
int wrcu_timer_end(wrcu_ctx* ctx, float* elapsed_ms); /* synchronises */

/* Profiling aid: while enabled, every draw brackets its RASTER kernel(s) (the vertex-stage setup
 * kernel excluded) with CUDA events on the context's stream; wrcu_last_raster_ms synchronises and
 * returns the duration of the most recent draw's raster work.  Used by bench.py's roofline lines. */
int wrcu_profile_enable(wrcu_ctx* ctx, int on);
int wrcu_last_raster_ms(wrcu_ctx* ctx, float* elapsed_ms);

/* Raw device pointer + pitch of a texture (GetColorBuffer, gl.cc:2317): valid
 * until the texture is destroyed.  Used by the multi-GPU tile gather. */
int wrcu_texture_device_ptr(wrcu_ctx* ctx, wrcu_tex tex, void** dptr,
                            size_t* pitch_bytes);
/* The CUDA stream (cudaStream_t) the context queues work on. */
int wrcu_stream(wrcu_ctx* ctx, void** stream);

/* ---- software-compositor blit ------------------------------------------------------------------
 * `Composite` of the SWGL surface (swgl/src/composite.h:532-590), the call Gecko's SwCompositor
 * (compositor/sw_compositor.rs) makes per tile: the `src_rect` (x, y, w, h) of one RGBA8 texture into
 * the `dst_rect` of another, clipped to `clip_rect` (destination space) — integer-ratio nearest
 * scaling (scale_blit, composite.h:166-282) or, when flipped in x or when the sizes differ under a
 * LINEAR filter (and the source is at least 2 texels wide), the 7-bit bilinear filter (linear_blit,
 * composite.h:353-417); `opaque` copies, otherwise premultiplied-alpha over.  Bit-exact with the
 * reference's row walkers, including their per-chunk float running sums. */
int wrcu_composite_blit(wrcu_ctx* ctx, wrcu_tex dst, wrcu_tex src,
                        const int32_t src_rect[4], const int32_t dst_rect[4],
                        int opaque, int flip_x, int flip_y, int filter_linear,
                        const int32_t clip_rect[4]);

/* `CompositeYUV` of the SWGL surface (swgl/src/composite.h:1335-1384; compositor/sw_compositor.rs composites video
 * surfaces with it): three planes (R8 textures at `color_depth` 8, or LSB-aligned R16 textures at `color_depth`
 * 10, 12 or 16; the two chroma planes of one size, full or half resolution)
 * converted to BGRA with the 6/7-bit fixed-point matrix of `color_space` (YUVRangedColorSpace, composite.h:1210-1218:
 * 0 BT601 narrow, 1 BT601 full, 2 BT709 narrow, 3 BT709 full, 4 BT2020 narrow, 5 BT2020 full, 6 GBR identity) while the
 * `src_rect` of the luma plane is scaled into `dst_rect` with the reference's row walker (linear_row_yuv: integer
 * coordinates, the half-resolution-chroma upscale path of 8-bit planes included), clipped to `clip_rect`; opaque.
 * Bit-exact.  The matrix is the 8-bit one at every depth, as in the reference.  Any other plane format / depth
 * combination, and planes under 2 texels wide, give WRCU_ERR_UNSUPPORTED. */
int wrcu_composite_blit_yuv(wrcu_ctx* ctx, wrcu_tex dst, wrcu_tex y_plane, wrcu_tex u_plane, wrcu_tex v_plane,
                            int color_space, uint32_t color_depth,
                            const int32_t src_rect[4], const int32_t dst_rect[4],
                            int flip_x, int flip_y, const int32_t clip_rect[4]);

/* ---- multi-GPU: the tiles of ONE frame sharded over GPUs (SURVEY.md §8e) ----------------------
 * Picture-cache tiles are independent render targets (frame_builder.rs:995-1057): each GPU draws its
 * share with no data-path communication.  The one exchange step — finished tiles into the
 * framebuffer that is presented — needs no collective and no staging either: the compositing GPU
 * EXPORTS its framebuffer texture, every other context IMPORTS it (CUDA IPC between processes, the
 * raw mapping inside one process; peer access over NVLink / NVSwitch) and binds it as the target of
 * its own `composite` tile list, so the copy kernel's bulk-tensor stores land in the remote
 * framebuffer directly.  Ordering between contexts is by flag words in device memory, written and
 * polled on the CUDA streams — no host synchronisation per frame.
 * One process per GPU (torchrun) or several contexts in one process both work. */
typedef struct wrcu_ipc_texture {
  uint8_t handle[64];          /* cudaIpcMemHandle_t                                  */
  uint64_t pid, address;       /* exporting process and its device address            */
  uint64_t pitch;
  int32_t format, width, height, device;
} wrcu_ipc_texture;
int wrcu_texture_export(wrcu_ctx* ctx, wrcu_tex tex, wrcu_ipc_texture* out);
/* The imported texture aliases the exporter's memory: usable as a render target or sampler
 * source; wrcu_texture_destroy unmaps it. */
int wrcu_texture_import(wrcu_ctx* ctx, const wrcu_ipc_texture* in, wrcu_tex* out);
typedef struct wrcu_ipc_flags {
  uint8_t handle[64];
  uint64_t pid, address;
  int32_t count, device;
} wrcu_ipc_flags;
/* This context's flag words (`count` x u32 in device memory, zeroed); `out` is what peers open. */
int wrcu_peer_flags_create(wrcu_ctx* ctx, int count, wrcu_ipc_flags* out);
/* Map a peer's flag words; *peer_id identifies it in wrcu_peer_signal. */
int wrcu_peer_flags_open(wrcu_ctx* ctx, const wrcu_ipc_flags* in, int* peer_id);
/* Stream-ordered: once everything queued on this context so far has completed (its stores to
 * imported textures included), peer.flags[slot] = value. */
int wrcu_peer_signal(wrcu_ctx* ctx, int peer_id, int slot, uint32_t value);
/* Stream-ordered: work queued on this context after the call starts only when this context's own
 * flags[slot] >= value (wrap-safe).  A peer that never signals is reported after ~2 s as
 * WRCU_ERR_CUDA at the next synchronisation instead of hanging the GPU. */
int wrcu_peer_wait(wrcu_ctx* ctx, int slot, uint32_t value);

/* ---- asynchronous readback (the reference's PBO path) ----------------------- */
/* Page-locked host memory for uploads/readbacks: create_pbo_with_size /
 * map_pbo_for_readback (device/gl.rs:3146, 3241).  Buffers from here make
 * wrcu_texture_upload / wrcu_read_pixels[_async] run at full PCIe rate. */
int wrcu_host_alloc(wrcu_ctx* ctx, size_t bytes, void** out);
int wrcu_host_free(wrcu_ctx* ctx, void* ptr);
/* read_pixels_into_pbo (device/gl.rs:3190): queue a readback of `tex` behind
 * the draws issued so far and return at once; the copy runs on a second stream,
 * so it overlaps the following draws (which must target another texture — a
 * later wrcu_target_bind of `tex` waits for the copy).  `*fence` identifies the
 * copy; `out` is valid after wrcu_fence_wait(fence) or wrcu_finish. */
int wrcu_read_pixels_async(wrcu_ctx* ctx, wrcu_tex tex, int x, int y, int w,
                           int h, void* out, size_t dst_stride, uint64_t* fence);
int wrcu_fence_wait(wrcu_ctx* ctx, uint64_t fence);
/* glFenceSync (device/gl.rs:3243 insert_fence_sync via UploadPBOPool, renderer/upload.rs:449-470):
 * a fence behind everything queued so far.  Ownership rule for page-locked upload buffers: a
 * wrcu_host_alloc buffer passed to wrcu_texture_upload / wrcu_texture_upload_batch is read by the
 * GPU in place (no intermediate copy) and stays BUSY until a fence inserted after the call has been
 * waited on (or wrcu_finish) — exactly how the reference recycles its upload PBOs.  Every other
 * array (instances, tables, texture lists, GPU-cache blocks) is copied before the call returns. */
int wrcu_fence_insert(wrcu_ctx* ctx, uint64_t* fence);

#ifdef __cplusplus
}
#endif
#endif /* WRCU_H */
