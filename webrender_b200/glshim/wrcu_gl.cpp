// wrcu_gl.cpp — the reference's OWN FFI surface over the wrcu backend.
//
// WebRender reaches its software rasteriser through `impl Gl for swgl::Context`, which
// forwards to the `extern "C"` symbols declared in swgl/src/swgl_fns.rs:23-320 and defined in
// swgl/src/gl.cc:1080-2851 (+ composite.h).  This library exports the SAME symbols with the
// same signatures; behind them a small GL state machine (textures, buffers, VAOs, FBOs,
// programs selected by name string, blend/depth/scissor state) turns every
// DrawElementsInstanced / Clear / ReadPixels / TexSubImage2D into calls on include/wrcu.h.
// A host linked against it instead of SWGL needs no source change (SURVEY.md §8b, option 1).
//
// Scope: the calls `Device` issues on the frame-draw path and its update path, and the software
// compositor's hooks (LockTexture / LockFramebuffer / Composite / CompositeYUV / GetResourceBuffer) as
// device-side blits.  SetTextureBuffer (a caller-owned CPU buffer as texture storage) has no
// counterpart for device memory: it sets GL_INVALID_OPERATION.
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/wrcu.h"

typedef unsigned int GLenum;
typedef unsigned int GLuint;
typedef int GLint;
typedef int GLsizei;
typedef unsigned int GLbitfield;
typedef unsigned char GLboolean;
typedef float GLfloat;
typedef double GLdouble;
typedef char GLchar;
typedef void GLvoid;
typedef intptr_t GLintptr;
typedef intptr_t GLsizeiptr;
typedef uint64_t GLuint64;

// swgl/src/gl_defs.h (standard GL values)
enum {
  GL_NO_ERROR = 0, GL_INVALID_ENUM = 0x0500, GL_INVALID_VALUE = 0x0501, GL_INVALID_OPERATION = 0x0502,
  GL_OUT_OF_MEMORY = 0x0505,
  GL_RGBA32F = 0x8814, GL_RGBA8 = 0x8058, GL_R8 = 0x8229, GL_RG8 = 0x822B, GL_R16 = 0x822A, GL_RG16 = 0x822C, GL_RG = 0x8227, GL_RGBA32I = 0x8D82, GL_DEPTH_COMPONENT24 = 0x81A6,
  GL_DEPTH_COMPONENT16 = 0x81A5, GL_DEPTH_COMPONENT32 = 0x81A7, GL_BGRA8 = 0x93A1,
  GL_BYTE = 0x1400, GL_UNSIGNED_BYTE = 0x1401, GL_SHORT = 0x1402, GL_UNSIGNED_SHORT = 0x1403, GL_INT = 0x1404, GL_FLOAT = 0x1406,
  GL_RED = 0x1903, GL_RGBA = 0x1908, GL_RGBA_INTEGER = 0x8D99, GL_BGRA = 0x80E1,
  GL_ARRAY_BUFFER = 0x8892, GL_ELEMENT_ARRAY_BUFFER = 0x8893, GL_PIXEL_PACK_BUFFER = 0x88EB,
  GL_PIXEL_UNPACK_BUFFER = 0x88EC,
  GL_FRAMEBUFFER = 0x8D40, GL_READ_FRAMEBUFFER = 0x8CA8, GL_DRAW_FRAMEBUFFER = 0x8CA9,
  GL_COLOR_ATTACHMENT0 = 0x8CE0, GL_DEPTH_ATTACHMENT = 0x8D00, GL_FRAMEBUFFER_COMPLETE = 0x8CD5,
  GL_RENDERBUFFER = 0x8D41,
  GL_COLOR_BUFFER_BIT = 0x4000, GL_DEPTH_BUFFER_BIT = 0x100,
  GL_NEAREST = 0x2600, GL_LINEAR = 0x2601, GL_TEXTURE_MAG_FILTER = 0x2800, GL_TEXTURE_MIN_FILTER = 0x2801,
  GL_TEXTURE_2D = 0x0DE1, GL_TEXTURE_RECTANGLE = 0x84F5, GL_TEXTURE0 = 0x84C0,
  GL_BLEND = 0x0BE2, GL_DEPTH_TEST = 0x0B71, GL_SCISSOR_TEST = 0x0C11, GL_TRIANGLES = 4,
  GL_ZERO = 0, GL_ONE = 1, GL_SRC_COLOR = 0x300, GL_ONE_MINUS_SRC_COLOR = 0x301, GL_SRC_ALPHA = 0x302,
  GL_ONE_MINUS_SRC_ALPHA = 0x303, GL_DST_ALPHA = 0x304, GL_ONE_MINUS_DST_ALPHA = 0x305, GL_DST_COLOR = 0x306,
  GL_ONE_MINUS_DST_COLOR = 0x307, GL_CONSTANT_COLOR = 0x8001, GL_ONE_MINUS_CONSTANT_COLOR = 0x8002,
  GL_CONSTANT_ALPHA = 0x8003, GL_ONE_MINUS_CONSTANT_ALPHA = 0x8004, GL_SRC1_ALPHA = 0x8589, GL_SRC1_COLOR = 0x88F9,
  GL_ONE_MINUS_SRC1_COLOR = 0x88FA, GL_ONE_MINUS_SRC1_ALPHA = 0x88FB,
  GL_FUNC_ADD = 0x8006, GL_MIN = 0x8007, GL_MAX = 0x8008, GL_MULTIPLY_KHR = 0x9294, GL_HSL_LUMINOSITY_KHR = 0x92B0,
  GL_LESS = 0x201, GL_LEQUAL = 0x203, GL_ALWAYS = 0x207,
  GL_UNPACK_ROW_LENGTH = 0x0CF2, GL_PACK_ROW_LENGTH = 0x0D02,
  GL_VENDOR = 0x1F00, GL_RENDERER = 0x1F01, GL_VERSION = 0x1F02, GL_EXTENSIONS = 0x1F03,
  GL_SHADING_LANGUAGE_VERSION = 0x8B8C,
  GL_MAX_TEXTURE_SIZE = 0x0D33, GL_MAX_TEXTURE_UNITS = 0x84E2, GL_MAX_TEXTURE_IMAGE_UNITS = 0x8872,
  GL_MAX_ARRAY_TEXTURE_LAYERS = 0x88FF, GL_READ_FRAMEBUFFER_BINDING = 0x8CAA, GL_DRAW_FRAMEBUFFER_BINDING = 0x8CA6,
  GL_PIXEL_PACK_BUFFER_BINDING = 0x88ED, GL_PIXEL_UNPACK_BUFFER_BINDING = 0x88EF, GL_NUM_EXTENSIONS = 0x821D,
  GL_MAJOR_VERSION = 0x821B, GL_MINOR_VERSION = 0x821C, GL_MIN_PROGRAM_TEXEL_OFFSET = 0x8904,
  GL_MAX_PROGRAM_TEXEL_OFFSET = 0x8905, GL_DEPTH_WRITEMASK = 0x0B72,
  GL_QUERY_RESULT = 0x8866, GL_QUERY_RESULT_AVAILABLE = 0x8867,
};

namespace {

struct Tex {
  bool live = false;
  GLenum ifmt = 0;
  int w = 0, h = 0;
  int filter = GL_NEAREST;
  wrcu_tex dev = 0;             // RGBA8 / R8 / DEPTH24: a wrcu texture
  std::vector<uint8_t> shadow;  // RGBA32F / RGBA32I data textures: host copy handed to wrcu_frame_begin
  uint64_t version = 0;
};
struct Buf { std::vector<uint8_t> data; };
struct Attr {
  bool enabled = false, integer = false, normalized = false;
  GLuint buf = 0;
  int size = 0, stride = 0, divisor = 0;
  GLenum type = 0;
  size_t offset = 0;
};
struct Vao { Attr a[16]; GLuint ibo = 0; };
struct Fbo { GLuint color = 0, depth_tex = 0, depth_rb = 0; };
struct Rb { wrcu_tex dev = 0; int w = 0, h = 0; };
static const char* const kSamplers[12] = {"sColor0", "sColor1", "sColor2", "sGpuCache", "sTransformPalette",
                                          "sRenderTasks", "sDither", "sPrimitiveHeadersF", "sPrimitiveHeadersI",
                                          "sClipMask", "sGpuBufferF", "sGpuBufferI"};
enum { LOC_UTRANSFORM = 100, LOC_UMODE = 101 };
struct Prog {
  std::string name;
  bool linked = false;
  int kind = 0;
  uint32_t feats = 0;
  int slot[12];
  float uTransform[16];
  Prog() {
    for (int i = 0; i < 12; i++) slot[i] = i;  // the fixed slots of renderer/mod.rs:369-386
    memset(uTransform, 0, sizeof uTransform);
    uTransform[0] = uTransform[5] = uTransform[10] = uTransform[15] = 1.0f;
  }
};

struct Context {
  wrcu_ctx* dev = nullptr;
  int refs = 1;
  GLenum error = GL_NO_ERROR;
  std::map<GLuint, Tex> tex;
  std::map<GLuint, Buf> buf;
  std::map<GLuint, Vao> vao;
  std::map<GLuint, Fbo> fbo;
  std::map<GLuint, Rb> rb;
  std::map<GLuint, Prog> prog;
  std::map<GLuint, std::string> shader;
  GLuint next_id = 1;
  // bindings
  int active_unit = 0;
  GLuint unit_tex[16] = {0};
  GLuint array_buffer = 0, pack_buffer = 0, unpack_buffer = 0;
  GLuint cur_vao = 0, draw_fbo = 0, read_fbo = 0, cur_rb = 0, cur_prog = 0;
  // state
  bool blend = false, depth_test = false, scissor_test = false;
  GLenum srgb = GL_ONE, drgb = GL_ZERO, sa = GL_ONE, da = GL_ZERO, equation = GL_FUNC_ADD, depth_func = GL_LESS;
  float blend_color[4] = {0, 0, 0, 0};
  bool depth_mask = true;
  int scissor[4] = {0, 0, 0, 0}, viewport[4] = {0, 0, 0, 0};
  float clear_color[4] = {0, 0, 0, 0};
  double clear_depth = 1.0;
  int unpack_row_length = 0, pack_row_length = 0;
  // frame tables last handed to wrcu_frame_begin: (texture id, version) per table sampler
  bool in_frame = false;
  GLuint table_tex[7] = {0};
  uint64_t table_ver[7] = {0};
  // target last bound
  GLuint bound_color = 0;
  wrcu_tex bound_depth = 0;
  float bound_proj[16] = {0};
  int bound_vp[4] = {0, 0, 0, 0};
  bool target_valid = false;
  Vao vao0;
};
Context* ctx = nullptr;

void set_error(GLenum e) { if (ctx && ctx->error == GL_NO_ERROR) ctx->error = e; }
void check(int rc) {
  if (rc == WRCU_OK) return;
  set_error(rc == WRCU_ERR_OOM ? GL_OUT_OF_MEMORY : GL_INVALID_OPERATION);
}
Tex* tex_of(GLuint id) {
  auto it = ctx->tex.find(id);
  return it == ctx->tex.end() || !it->second.live ? nullptr : &it->second;
}
Vao& cur_vao() { return ctx->cur_vao ? ctx->vao[ctx->cur_vao] : ctx->vao0; }
int wr_fmt(GLenum ifmt) {
  switch (ifmt) {
    case GL_RGBA8: case GL_BGRA8: return WRCU_FMT_RGBA8;
    case GL_R8: return WRCU_FMT_R8;
    case GL_RG8: return WRCU_FMT_RG8;
    case GL_R16: return WRCU_FMT_R16;
    case GL_RG16: return WRCU_FMT_RG16;
    case GL_DEPTH_COMPONENT24: case GL_DEPTH_COMPONENT16: case GL_DEPTH_COMPONENT32: return WRCU_FMT_DEPTH24;
    default: return 0;
  }
}
int bytes_per_pixel(GLenum ifmt) {
  switch (ifmt) {
    case GL_RGBA8: case GL_BGRA8: return 4;
    case GL_R8: return 1;
    case GL_RG8: case GL_R16: return 2;
    case GL_RG16: return 4;
    case GL_RGBA32F: case GL_RGBA32I: return 16;
    default: return 4;
  }
}
void storage(Tex& t, GLenum ifmt, int w, int h) {
  if (t.dev) { wrcu_texture_destroy(ctx->dev, t.dev); t.dev = 0; }
  t.live = true;
  t.ifmt = ifmt;
  t.w = w;
  t.h = h;
  t.shadow.clear();
  t.version++;
  if (ifmt == GL_RGBA32F || ifmt == GL_RGBA32I) {
    t.shadow.assign((size_t)w * h * 16, 0);
  } else if (int f = wr_fmt(ifmt)) {
    check(wrcu_texture_create(ctx->dev, f, w, h, &t.dev));
    if (t.dev && f != WRCU_FMT_DEPTH24) wrcu_texture_set_filter(ctx->dev, t.dev, t.filter == GL_LINEAR ? WRCU_LINEAR : WRCU_NEAREST);
  } else {
    set_error(GL_INVALID_ENUM);
  }
  ctx->target_valid = false;
}
Fbo* fbo_of(GLuint id) {
  auto it = ctx->fbo.find(id);
  return it == ctx->fbo.end() ? nullptr : &it->second;
}
// colour and depth of a framebuffer object as wrcu textures
bool fbo_attachments(GLuint id, Tex** color, wrcu_tex* depth) {
  Fbo* f = fbo_of(id);
  if (!f) return false;
  *color = tex_of(f->color);
  *depth = 0;
  if (f->depth_tex) { if (Tex* d = tex_of(f->depth_tex)) *depth = d->dev; }
  else if (f->depth_rb) { auto it = ctx->rb.find(f->depth_rb); if (it != ctx->rb.end()) *depth = it->second.dev; }
  return *color != nullptr && (*color)->dev != 0;
}
bool bind_target(GLuint fbo_id, const float* proj) {
  Tex* color = nullptr;
  wrcu_tex depth = 0;
  if (!fbo_attachments(fbo_id, &color, &depth)) { set_error(GL_INVALID_OPERATION); return false; }
  GLuint cid = fbo_of(fbo_id)->color;
  if (ctx->target_valid && ctx->bound_color == cid && ctx->bound_depth == depth &&
      !memcmp(ctx->bound_proj, proj, sizeof ctx->bound_proj) && !memcmp(ctx->bound_vp, ctx->viewport, sizeof ctx->bound_vp))
    return true;
  int vp[4] = {ctx->viewport[0], ctx->viewport[1], ctx->viewport[2], ctx->viewport[3]};
  if (vp[2] <= 0 || vp[3] <= 0) { vp[0] = vp[1] = 0; vp[2] = color->w; vp[3] = color->h; }
  int rc = wrcu_target_bind(ctx->dev, color->dev, depth, proj, vp);
  check(rc);
  if (rc != WRCU_OK) return false;
  ctx->bound_color = cid;
  ctx->bound_depth = depth;
  memcpy(ctx->bound_proj, proj, sizeof ctx->bound_proj);
  memcpy(ctx->bound_vp, ctx->viewport, sizeof ctx->bound_vp);
  ctx->target_valid = true;
  return true;
}

// hash_blend_key (gl.cc:1287-1315) onto the wrcu_blend enumeration
GLenum remap_blendfunc(GLenum rgb, GLenum a) {
  switch (a) {
    case GL_SRC_ALPHA: if (rgb == GL_SRC_COLOR) a = GL_SRC_COLOR; break;
    case GL_ONE_MINUS_SRC_ALPHA: if (rgb == GL_ONE_MINUS_SRC_COLOR) a = GL_ONE_MINUS_SRC_COLOR; break;
    case GL_DST_ALPHA: if (rgb == GL_DST_COLOR) a = GL_DST_COLOR; break;
    case GL_ONE_MINUS_DST_ALPHA: if (rgb == GL_ONE_MINUS_DST_COLOR) a = GL_ONE_MINUS_DST_COLOR; break;
    case GL_CONSTANT_ALPHA: if (rgb == GL_CONSTANT_COLOR) a = GL_CONSTANT_COLOR; break;
    case GL_ONE_MINUS_CONSTANT_ALPHA: if (rgb == GL_ONE_MINUS_CONSTANT_COLOR) a = GL_ONE_MINUS_CONSTANT_COLOR; break;
    case GL_SRC_COLOR: if (rgb == GL_SRC_ALPHA) a = GL_SRC_ALPHA; break;
    case GL_ONE_MINUS_SRC_COLOR: if (rgb == GL_ONE_MINUS_SRC_ALPHA) a = GL_ONE_MINUS_SRC_ALPHA; break;
    case GL_DST_COLOR: if (rgb == GL_DST_ALPHA) a = GL_DST_ALPHA; break;
    case GL_ONE_MINUS_DST_COLOR: if (rgb == GL_ONE_MINUS_DST_ALPHA) a = GL_ONE_MINUS_DST_ALPHA; break;
    case GL_CONSTANT_COLOR: if (rgb == GL_CONSTANT_ALPHA) a = GL_CONSTANT_ALPHA; break;
    case GL_ONE_MINUS_CONSTANT_COLOR: if (rgb == GL_ONE_MINUS_CONSTANT_ALPHA) a = GL_ONE_MINUS_CONSTANT_ALPHA; break;
    case GL_SRC1_ALPHA: if (rgb == GL_SRC1_COLOR) a = GL_SRC1_COLOR; break;
    case GL_ONE_MINUS_SRC1_ALPHA: if (rgb == GL_ONE_MINUS_SRC1_COLOR) a = GL_ONE_MINUS_SRC1_COLOR; break;
    case GL_SRC1_COLOR: if (rgb == GL_SRC1_ALPHA) a = GL_SRC1_ALPHA; break;
    case GL_ONE_MINUS_SRC1_COLOR: if (rgb == GL_ONE_MINUS_SRC1_ALPHA) a = GL_ONE_MINUS_SRC1_ALPHA; break;
  }
  return a;
}
int blend_key() {
  if (!ctx->blend) return WRCU_BLEND_NONE;
  const GLenum eq = ctx->equation;
  if (eq != GL_FUNC_ADD) {
    if (eq == GL_MIN) return WRCU_BLEND_MIN;
    if (eq == GL_MAX) return WRCU_BLEND_MAX;
    // KHR_blend_equation_advanced, in FOR_EACH_BLEND_KEY's order (gl.cc:631-645)
    static const GLenum adv[15] = {0x9294, 0x9295, 0x9296, 0x9297, 0x9298, 0x9299, 0x929A, 0x929B,
                                   0x929C, 0x929E, 0x92A0, 0x92AD, 0x92AE, 0x92AF, 0x92B0};
    for (int i = 0; i < 15; i++) if (adv[i] == eq) return WRCU_BLEND_ADV_MULTIPLY + i;
    return -1;
  }
  const GLenum s = ctx->srgb, d = ctx->drgb;
  const bool separate = s != ctx->sa || d != ctx->da;
  struct K { GLenum s, d, sa, da; int key; };
  static const K keys[] = {
      {GL_ONE, GL_ZERO, 0, 0, WRCU_BLEND_NONE},
      {GL_SRC_ALPHA, GL_ONE_MINUS_SRC_ALPHA, GL_ONE, GL_ONE_MINUS_SRC_ALPHA, WRCU_BLEND_ALPHA},
      {GL_ONE, GL_ONE_MINUS_SRC_ALPHA, 0, 0, WRCU_BLEND_PREMULTIPLIED_ALPHA},
      {GL_ZERO, GL_ONE_MINUS_SRC_COLOR, 0, 0, WRCU_BLEND_SUBPIXEL_PASS0},
      {GL_ZERO, GL_ONE_MINUS_SRC_COLOR, GL_ZERO, GL_ONE, WRCU_BLEND_SUBPIXEL_PASS0_KEEP_A},
      {GL_ZERO, GL_ONE_MINUS_SRC_ALPHA, 0, 0, WRCU_BLEND_PREMULTIPLIED_DEST_OUT},
      {GL_ZERO, GL_SRC_COLOR, 0, 0, WRCU_BLEND_MULTIPLY},
      {GL_ONE, GL_ONE, 0, 0, WRCU_BLEND_PLUS_LIGHTER},
      {GL_ONE, GL_ONE, GL_ONE, GL_ONE_MINUS_SRC_ALPHA, WRCU_BLEND_ADD_KEEP_ALPHA_OVER},
      {GL_ONE_MINUS_DST_ALPHA, GL_ONE, GL_ZERO, GL_ONE, WRCU_BLEND_DST_ALPHA_ADD},
      {GL_CONSTANT_COLOR, GL_ONE_MINUS_SRC_COLOR, 0, 0, WRCU_BLEND_CONSTANT_COLOR},
      {GL_ONE, GL_ONE_MINUS_SRC1_COLOR, 0, 0, WRCU_BLEND_SUBPIXEL_DUAL_SOURCE},
  };
  for (const K& k : keys) {
    if (k.s != s || k.d != d) continue;
    if (!separate && k.sa == 0 && k.da == 0) return k.key;
    if (separate && k.sa == ctx->sa && k.da == ctx->da && (k.sa || k.da)) return k.key;
  }
  return -1;
}

const void* table_ptr(int sampler, size_t* texels, GLuint* id, uint64_t* ver) {
  *texels = 0;
  *id = 0;
  *ver = 0;
  Prog& p = ctx->prog[ctx->cur_prog];
  int unit = p.slot[sampler];
  if (unit < 0 || unit >= 16) return nullptr;
  Tex* t = tex_of(ctx->unit_tex[unit]);
  if (!t || t->shadow.empty()) return nullptr;
  *texels = (size_t)t->w * t->h;
  *id = ctx->unit_tex[unit];
  *ver = t->version;
  return t->shadow.data();
}
// bind_frame_data: hand the bound data textures to the backend when any of them changed
bool sync_tables() {
  static const int samplers[7] = {7, 8, 4, 5, 3, 10, 11};  // prim_headers_f/i, transforms, render_tasks, gpu_cache, gpu_buffer_f/i
  wrcu_frame_tables t;
  memset(&t, 0, sizeof t);
  const void* ptr[7];
  size_t n[7];
  GLuint id[7];
  uint64_t ver[7];
  bool dirty = !ctx->in_frame;
  for (int i = 0; i < 7; i++) {
    ptr[i] = table_ptr(samplers[i], &n[i], &id[i], &ver[i]);
    if (id[i] != ctx->table_tex[i] || ver[i] != ctx->table_ver[i]) dirty = true;
  }
  if (!dirty) return true;
  if (ctx->in_frame) check(wrcu_frame_end(ctx->dev));
  t.prim_headers_f = (const float*)ptr[0]; t.prim_headers_f_texels = n[0];
  t.prim_headers_i = (const int32_t*)ptr[1]; t.prim_headers_i_texels = n[1];
  t.transforms = (const float*)ptr[2]; t.transforms_texels = n[2];
  t.render_tasks = (const float*)ptr[3]; t.render_tasks_texels = n[3];
  t.gpu_cache = (const float*)ptr[4]; t.gpu_cache_texels = n[4];
  t.gpu_buffer_f = (const float*)ptr[5]; t.gpu_buffer_f_texels = n[5];
  t.gpu_buffer_i = (const int32_t*)ptr[6]; t.gpu_buffer_i_texels = n[6];
  int rc = wrcu_frame_begin(ctx->dev, &t);
  check(rc);
  ctx->in_frame = rc == WRCU_OK;
  for (int i = 0; i < 7; i++) { ctx->table_tex[i] = id[i]; ctx->table_ver[i] = ver[i]; }
  return rc == WRCU_OK;
}
GLuint gen_id() { return ctx->next_id++; }
Buf* bound_buffer(GLenum target) {
  GLuint id = 0;
  switch (target) {
    case GL_ARRAY_BUFFER: id = ctx->array_buffer; break;
    case GL_ELEMENT_ARRAY_BUFFER: id = cur_vao().ibo; break;
    case GL_PIXEL_PACK_BUFFER: id = ctx->pack_buffer; break;
    case GL_PIXEL_UNPACK_BUFFER: id = ctx->unpack_buffer; break;
    default: return nullptr;
  }
  if (!id) return nullptr;
  return &ctx->buf[id];
}
// upload rows of a (possibly PBO-sourced) client image into a texture
void upload(Tex& t, int x, int y, int w, int h, GLenum format, const void* data) {
  const int bpp = bytes_per_pixel(t.ifmt);
  const uint8_t* src = (const uint8_t*)data;
  if (ctx->unpack_buffer) {
    Buf& b = ctx->buf[ctx->unpack_buffer];
    if ((size_t)(uintptr_t)data > b.data.size()) { set_error(GL_INVALID_OPERATION); return; }
    src = b.data.data() + (size_t)(uintptr_t)data;
  }
  if (!src || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > t.w || y + h > t.h) { set_error(GL_INVALID_VALUE); return; }
  const size_t src_stride = (size_t)(ctx->unpack_row_length > 0 ? ctx->unpack_row_length : w) * bpp;
  if (ctx->unpack_buffer) {  // the whole source image must lie inside the PBO
    const size_t off = (size_t)(uintptr_t)data, need = (size_t)(h - 1) * src_stride + (size_t)w * bpp;
    if (off + need > ctx->buf[ctx->unpack_buffer].data.size()) { set_error(GL_INVALID_OPERATION); return; }
  }
  if (!t.shadow.empty()) {
    for (int r = 0; r < h; r++)
      memcpy(t.shadow.data() + ((size_t)(y + r) * t.w + x) * 16, src + (size_t)r * src_stride, (size_t)w * 16);
    t.version++;
    return;
  }
  if (!t.dev) { set_error(GL_INVALID_OPERATION); return; }
  if (t.ifmt != GL_R8 && format == GL_RGBA) {
    // the backend stores BGRA like the reference (TextureFormat::RGBA8, gl.cc:1794-1836 swizzles on upload)
    std::vector<uint8_t> tmp((size_t)w * h * 4);
    for (int r = 0; r < h; r++) {
      const uint8_t* s = src + (size_t)r * src_stride;
      uint8_t* d = tmp.data() + (size_t)r * w * 4;
      for (int i = 0; i < w; i++) { d[4 * i] = s[4 * i + 2]; d[4 * i + 1] = s[4 * i + 1]; d[4 * i + 2] = s[4 * i]; d[4 * i + 3] = s[4 * i + 3]; }
    }
    check(wrcu_texture_upload(ctx->dev, t.dev, x, y, w, h, tmp.data(), (size_t)w * 4));
    return;
  }
  check(wrcu_texture_upload(ctx->dev, t.dev, x, y, w, h, src, src_stride));
}
void clear_rect(GLuint fbo_id, const int* rect, const float* color, const float* depth) {
  Prog ident;
  const float* proj = ctx->cur_prog ? ctx->prog[ctx->cur_prog].uTransform : ident.uTransform;
  if (!bind_target(fbo_id, proj)) return;
  check(wrcu_clear(ctx->dev, rect, color, depth));
}

}  // namespace

extern "C" {

// ---- context (gl.cc:2806-2851) ------------------------------------------------------------------
void* CreateContext() {
  Context* c = new Context();
  if (wrcu_ctx_create(0, &c->dev) != WRCU_OK) { delete c; return nullptr; }
  c->fbo[0] = Fbo();
  return c;
}
void ReferenceContext(void* c) { if (c) ((Context*)c)->refs++; }
void DestroyContext(void* p) {
  Context* c = (Context*)p;
  if (!c || --c->refs > 0) return;
  if (ctx == c) ctx = nullptr;
  wrcu_ctx_destroy(c->dev);
  delete c;
}
void MakeCurrent(void* c) { ctx = (Context*)c; }
size_t ReportMemory(void*, size_t (*)(const void*)) { return 0; }

GLenum GetError() {
  GLenum e = ctx->error;
  if (e == GL_NO_ERROR) {
    int d = wrcu_get_error(ctx->dev);
    if (d == WRCU_ERR_OOM) e = GL_OUT_OF_MEMORY;
    else if (d != WRCU_OK) e = GL_INVALID_OPERATION;
  }
  ctx->error = GL_NO_ERROR;
  return e;
}
const char* GetString(GLenum name) {
  switch (name) {
    case GL_VENDOR: return "Mozilla Gfx";
    case GL_RENDERER: return wrcu_get_string(0);  // "Software WebRender": the host keeps is_software batching
    case GL_VERSION: return "3.2";
    case GL_SHADING_LANGUAGE_VERSION: return "1.50";
    default: return nullptr;
  }
}
static const char* const kExtensions[] = {
    "GL_ARB_blend_func_extended", "GL_ARB_clear_texture", "GL_ARB_copy_image", "GL_ARB_draw_instanced",
    "GL_ARB_explicit_attrib_location", "GL_ARB_instanced_arrays", "GL_ARB_invalidate_subdata",
    "GL_ARB_texture_storage", "GL_EXT_timer_query", "GL_KHR_blend_equation_advanced",
    "GL_KHR_blend_equation_advanced_coherent"};
const char* GetStringi(GLenum name, GLuint index) {
  if (name != GL_EXTENSIONS || index >= sizeof(kExtensions) / sizeof(kExtensions[0])) return nullptr;
  return kExtensions[index];
}
void GetIntegerv(GLenum pname, GLint* params) {
  switch (pname) {
    case GL_MAX_TEXTURE_UNITS: case GL_MAX_TEXTURE_IMAGE_UNITS: params[0] = 16; break;
    case GL_MAX_TEXTURE_SIZE: params[0] = 1 << 15; break;
    case GL_MAX_ARRAY_TEXTURE_LAYERS: params[0] = 0; break;
    case GL_READ_FRAMEBUFFER_BINDING: params[0] = (GLint)ctx->read_fbo; break;
    case GL_DRAW_FRAMEBUFFER_BINDING: params[0] = (GLint)ctx->draw_fbo; break;
    case GL_PIXEL_PACK_BUFFER_BINDING: params[0] = (GLint)ctx->pack_buffer; break;
    case GL_PIXEL_UNPACK_BUFFER_BINDING: params[0] = (GLint)ctx->unpack_buffer; break;
    case GL_NUM_EXTENSIONS: params[0] = (GLint)(sizeof(kExtensions) / sizeof(kExtensions[0])); break;
    case GL_MAJOR_VERSION: params[0] = 3; break;
    case GL_MINOR_VERSION: params[0] = 2; break;
    case GL_MIN_PROGRAM_TEXEL_OFFSET: params[0] = 0; break;
    case GL_MAX_PROGRAM_TEXEL_OFFSET: params[0] = 8; break;
    default: params[0] = 0; set_error(GL_INVALID_ENUM); break;
  }
}
void GetBooleanv(GLenum pname, GLboolean* params) {
  if (pname == GL_DEPTH_WRITEMASK) params[0] = ctx->depth_mask;
  else { params[0] = 0; set_error(GL_INVALID_ENUM); }
}
void Finish() { check(wrcu_finish(ctx->dev)); }

// ---- object names -------------------------------------------------------------------------------
void GenTextures(int n, GLuint* r) { for (int i = 0; i < n; i++) { r[i] = gen_id(); ctx->tex[r[i]] = Tex(); } }
void GenBuffers(int n, GLuint* r) { for (int i = 0; i < n; i++) { r[i] = gen_id(); ctx->buf[r[i]] = Buf(); } }
void GenFramebuffers(int n, GLuint* r) { for (int i = 0; i < n; i++) { r[i] = gen_id(); ctx->fbo[r[i]] = Fbo(); } }
void GenRenderbuffers(int n, GLuint* r) { for (int i = 0; i < n; i++) { r[i] = gen_id(); ctx->rb[r[i]] = Rb(); } }
void GenVertexArrays(int n, GLuint* r) { for (int i = 0; i < n; i++) { r[i] = gen_id(); ctx->vao[r[i]] = Vao(); } }
void GenQueries(GLsizei n, GLuint* r) { for (int i = 0; i < n; i++) r[i] = gen_id(); }
void DeleteTexture(GLuint n) {
  auto it = ctx->tex.find(n);
  if (it == ctx->tex.end()) return;
  if (it->second.dev) wrcu_texture_destroy(ctx->dev, it->second.dev);
  ctx->tex.erase(it);
  for (int i = 0; i < 16; i++) if (ctx->unit_tex[i] == n) ctx->unit_tex[i] = 0;
  ctx->target_valid = false;
}
void DeleteRenderbuffer(GLuint n) {
  auto it = ctx->rb.find(n);
  if (it == ctx->rb.end()) return;
  if (it->second.dev) wrcu_texture_destroy(ctx->dev, it->second.dev);
  ctx->rb.erase(it);
  ctx->target_valid = false;
}
void DeleteFramebuffer(GLuint n) { if (n) ctx->fbo.erase(n); ctx->target_valid = false; }
void DeleteBuffer(GLuint n) { ctx->buf.erase(n); }
void DeleteVertexArray(GLuint n) { ctx->vao.erase(n); if (ctx->cur_vao == n) ctx->cur_vao = 0; }
void DeleteQuery(GLuint) {}
void DeleteShader(GLuint s) { ctx->shader.erase(s); }
void DeleteProgram(GLuint p) { ctx->prog.erase(p); if (ctx->cur_prog == p) ctx->cur_prog = 0; }

// ---- bindings -----------------------------------------------------------------------------------
void ActiveTexture(GLenum texture) { ctx->active_unit = (int)(texture - GL_TEXTURE0) & 15; }
void BindTexture(GLenum, GLuint texture) { ctx->unit_tex[ctx->active_unit] = texture; }
void BindBuffer(GLenum target, GLuint buffer) {
  switch (target) {
    case GL_ARRAY_BUFFER: ctx->array_buffer = buffer; break;
    case GL_ELEMENT_ARRAY_BUFFER: cur_vao().ibo = buffer; break;
    case GL_PIXEL_PACK_BUFFER: ctx->pack_buffer = buffer; break;
    case GL_PIXEL_UNPACK_BUFFER: ctx->unpack_buffer = buffer; break;
    default: set_error(GL_INVALID_ENUM); break;
  }
}
void BindVertexArray(GLuint vao) { ctx->cur_vao = vao; }
void BindFramebuffer(GLenum target, GLuint fb) {
  if (target == GL_FRAMEBUFFER) ctx->draw_fbo = ctx->read_fbo = fb;
  else if (target == GL_DRAW_FRAMEBUFFER) ctx->draw_fbo = fb;
  else if (target == GL_READ_FRAMEBUFFER) ctx->read_fbo = fb;
  else set_error(GL_INVALID_ENUM);
}
void BindRenderbuffer(GLenum, GLuint rb) { ctx->cur_rb = rb; }

// ---- buffers ------------------------------------------------------------------------------------
void BufferData(GLenum target, GLsizeiptr size, const GLvoid* data, GLenum) {
  Buf* b = bound_buffer(target);
  if (!b) { set_error(GL_INVALID_OPERATION); return; }
  b->data.resize((size_t)size);
  if (data && size) memcpy(b->data.data(), data, (size_t)size);
}
void BufferSubData(GLenum target, GLintptr offset, GLsizeiptr size, const GLvoid* data) {
  Buf* b = bound_buffer(target);
  if (!b || offset < 0 || (size_t)(offset + size) > b->data.size()) { set_error(GL_INVALID_VALUE); return; }
  memcpy(b->data.data() + offset, data, (size_t)size);
}
void* MapBuffer(GLenum target, GLbitfield) {
  Buf* b = bound_buffer(target);
  return b && !b->data.empty() ? b->data.data() : nullptr;
}
void* MapBufferRange(GLenum target, GLintptr offset, GLsizeiptr length, GLbitfield) {
  Buf* b = bound_buffer(target);
  if (!b || offset < 0 || (size_t)(offset + length) > b->data.size()) return nullptr;
  return b->data.data() + offset;
}
GLboolean UnmapBuffer(GLenum target) { return bound_buffer(target) != nullptr; }

// ---- textures -----------------------------------------------------------------------------------
void TexStorage2D(GLenum, GLint, GLenum internal_format, GLsizei width, GLsizei height) {
  GLuint id = ctx->unit_tex[ctx->active_unit];
  if (!id || width <= 0 || height <= 0) { set_error(GL_INVALID_OPERATION); return; }
  storage(ctx->tex[id], internal_format, width, height);
}
void TexImage2D(GLenum target, GLint level, GLint internal_format, GLsizei width, GLsizei height, GLint,
                GLenum format, GLenum, const GLvoid* data) {
  if (level != 0) return;
  TexStorage2D(target, 1, (GLenum)internal_format, width, height);
  GLuint id = ctx->unit_tex[ctx->active_unit];
  if (data && id && ctx->tex[id].live) upload(ctx->tex[id], 0, 0, width, height, format, data);
}
void TexSubImage2D(GLenum, GLint level, GLint xoffset, GLint yoffset, GLsizei width, GLsizei height, GLenum format,
                   GLenum, const GLvoid* data) {
  if (level != 0) return;
  Tex* t = tex_of(ctx->unit_tex[ctx->active_unit]);
  if (!t) { set_error(GL_INVALID_OPERATION); return; }
  upload(*t, xoffset, yoffset, width, height, format, data);
}
void GenerateMipmap(GLenum) {}
void SetTextureParameter(GLuint id, GLenum pname, GLint param) {
  Tex* t = nullptr;
  auto it = ctx->tex.find(id);
  if (it != ctx->tex.end()) t = &it->second;
  if (!t) { set_error(GL_INVALID_OPERATION); return; }
  if (pname == GL_TEXTURE_MAG_FILTER || pname == GL_TEXTURE_MIN_FILTER) {
    t->filter = param == GL_LINEAR ? GL_LINEAR : GL_NEAREST;
    if (t->dev && wr_fmt(t->ifmt) != WRCU_FMT_DEPTH24)
      check(wrcu_texture_set_filter(ctx->dev, t->dev, t->filter == GL_LINEAR ? WRCU_LINEAR : WRCU_NEAREST));
  }
}
void TexParameteri(GLenum, GLenum pname, GLint param) { SetTextureParameter(ctx->unit_tex[ctx->active_unit], pname, param); }
void PixelStorei(GLenum name, GLint param) {
  if (name == GL_UNPACK_ROW_LENGTH) ctx->unpack_row_length = param;
  else if (name == GL_PACK_ROW_LENGTH) ctx->pack_row_length = param;
}
void SetTextureBuffer(GLuint, GLenum, GLsizei, GLsizei, GLsizei, void*, GLsizei, GLsizei) {
  set_error(GL_INVALID_OPERATION);  // external CPU memory as texture storage: not for device textures
}

// ---- framebuffers -------------------------------------------------------------------------------
void FramebufferTexture2D(GLenum target, GLenum attachment, GLenum, GLuint texture, GLint) {
  GLuint id = target == GL_READ_FRAMEBUFFER ? ctx->read_fbo : ctx->draw_fbo;
  Fbo& f = ctx->fbo[id];
  if (attachment == GL_COLOR_ATTACHMENT0) f.color = texture;
  else if (attachment == GL_DEPTH_ATTACHMENT) { f.depth_tex = texture; f.depth_rb = 0; }
  else set_error(GL_INVALID_ENUM);
  ctx->target_valid = false;
}
void FramebufferRenderbuffer(GLenum target, GLenum attachment, GLenum, GLuint renderbuffer) {
  GLuint id = target == GL_READ_FRAMEBUFFER ? ctx->read_fbo : ctx->draw_fbo;
  Fbo& f = ctx->fbo[id];
  if (attachment == GL_DEPTH_ATTACHMENT) { f.depth_rb = renderbuffer; f.depth_tex = 0; }
  else set_error(GL_INVALID_ENUM);
  ctx->target_valid = false;
}
void RenderbufferStorage(GLenum, GLenum internalformat, GLsizei width, GLsizei height) {
  if (!ctx->cur_rb || wr_fmt(internalformat) != WRCU_FMT_DEPTH24) { set_error(GL_INVALID_OPERATION); return; }
  Rb& r = ctx->rb[ctx->cur_rb];
  if (r.dev) wrcu_texture_destroy(ctx->dev, r.dev);
  r.dev = 0;
  r.w = width;
  r.h = height;
  check(wrcu_texture_create(ctx->dev, WRCU_FMT_DEPTH24, width, height, &r.dev));
  ctx->target_valid = false;
}
GLenum CheckFramebufferStatus(GLenum) { return GL_FRAMEBUFFER_COMPLETE; }
void InvalidateFramebuffer(GLenum, GLsizei, const GLenum*) {}
void ResolveFramebuffer(GLuint) {}  // SWGL's delayed clears have no counterpart: clears are queued in order
void InitDefaultFramebuffer(int, int, int width, int height, int, void*) {
  // the default framebuffer (window) becomes a device texture of that size; the CPU buffer the
  // caller offers is not used (present = GetColorBuffer / ReadPixels)
  Fbo& f = ctx->fbo[0];
  if (!f.color) { f.color = gen_id(); ctx->tex[f.color] = Tex(); }
  Tex& t = ctx->tex[f.color];
  if (!t.live || t.w != width || t.h != height) storage(t, GL_RGBA8, width, height);
}
void* GetColorBuffer(GLuint, GLboolean, int32_t* width, int32_t* height, int32_t* stride) {
  if (width) *width = 0;
  if (height) *height = 0;
  if (stride) *stride = 0;
  set_error(GL_INVALID_OPERATION);  // device memory cannot be lent as a CPU pointer; use ReadPixels
  return nullptr;
}

// ---- programs -----------------------------------------------------------------------------------
GLuint CreateShader(GLenum) { GLuint id = gen_id(); ctx->shader[id] = std::string(); return id; }
void ShaderSourceByName(GLuint shader, const GLchar* name) { ctx->shader[shader] = name ? name : ""; }
GLuint CreateProgram() { GLuint id = gen_id(); ctx->prog[id] = Prog(); return id; }
void AttachShader(GLuint program, GLuint shader) {
  Prog& p = ctx->prog[program];
  p.name = ctx->shader[shader];
  // programs are selected by name string "<shader>[ FEAT,FEAT]" (swgl/build.rs:13-31, gl.cc:1431)
  p.linked = wrcu_program_from_name(p.name.c_str(), &p.kind, &p.feats) == WRCU_OK;
}
void LinkProgram(GLuint) {}
GLint GetLinkStatus(GLuint program) {
  auto it = ctx->prog.find(program);
  return it != ctx->prog.end() && it->second.linked ? 1 : 0;
}
void UseProgram(GLuint program) { ctx->cur_prog = program; }
void BindAttribLocation(GLuint, GLuint, const GLchar*) {}  // instance layouts are the kind's #[repr(C)] struct
GLint GetAttribLocation(GLuint, const GLchar*) { return -1; }
GLint GetUniformLocation(GLuint, const GLchar* name) {
  if (!name) return -1;
  if (!strcmp(name, "uTransform")) return LOC_UTRANSFORM;
  if (!strcmp(name, "uMode")) return LOC_UMODE;
  for (int i = 0; i < 12; i++) if (!strcmp(name, kSamplers[i])) return i;
  return -1;
}
void Uniform1i(GLint location, GLint v0) {
  if (!ctx->cur_prog) return;
  if (location >= 0 && location < 12) ctx->prog[ctx->cur_prog].slot[location] = v0;
}
void Uniform4fv(GLint, GLsizei, const GLfloat*) {}
void UniformMatrix4fv(GLint location, GLsizei, GLboolean, const GLfloat* value) {
  if (location == LOC_UTRANSFORM && ctx->cur_prog) memcpy(ctx->prog[ctx->cur_prog].uTransform, value, 64);
}

// ---- vertex arrays ------------------------------------------------------------------------------
void EnableVertexAttribArray(GLuint index) { if (index < 16) cur_vao().a[index].enabled = true; }
void VertexAttribDivisor(GLuint index, GLuint divisor) { if (index < 16) cur_vao().a[index].divisor = (int)divisor; }
void VertexAttribPointer(GLuint index, GLint size, GLenum type, GLboolean normalized, GLsizei stride, GLuint offset) {
  if (index >= 16) return;
  Attr& a = cur_vao().a[index];
  a.buf = ctx->array_buffer; a.size = size; a.type = type; a.normalized = normalized; a.stride = stride;
  a.offset = offset; a.integer = false;
}
void VertexAttribIPointer(GLuint index, GLint size, GLenum type, GLsizei stride, GLuint offset) {
  if (index >= 16) return;
  Attr& a = cur_vao().a[index];
  a.buf = ctx->array_buffer; a.size = size; a.type = type; a.normalized = false; a.stride = stride;
  a.offset = offset; a.integer = true;
}

// ---- fixed-function state -----------------------------------------------------------------------
void Enable(GLenum cap) {
  if (cap == GL_BLEND) ctx->blend = true;
  else if (cap == GL_DEPTH_TEST) ctx->depth_test = true;
  else if (cap == GL_SCISSOR_TEST) ctx->scissor_test = true;
}
void Disable(GLenum cap) {
  if (cap == GL_BLEND) ctx->blend = false;
  else if (cap == GL_DEPTH_TEST) ctx->depth_test = false;
  else if (cap == GL_SCISSOR_TEST) ctx->scissor_test = false;
}
void BlendFunc(GLenum srgb, GLenum drgb, GLenum sa, GLenum da) {
  ctx->srgb = srgb;
  ctx->drgb = drgb;
  ctx->sa = remap_blendfunc(srgb, sa);
  ctx->da = remap_blendfunc(drgb, da);
}
void BlendColor(GLfloat r, GLfloat g, GLfloat b, GLfloat a) {
  ctx->blend_color[0] = r; ctx->blend_color[1] = g; ctx->blend_color[2] = b; ctx->blend_color[3] = a;
}
void BlendEquation(GLenum mode) { ctx->equation = mode; }
void DepthMask(GLboolean flag) { ctx->depth_mask = flag != 0; }
void DepthFunc(GLenum func) { ctx->depth_func = func; }
void SetScissor(GLint x, GLint y, GLsizei w, GLsizei h) { ctx->scissor[0] = x; ctx->scissor[1] = y; ctx->scissor[2] = w; ctx->scissor[3] = h; }
void SetViewport(GLint x, GLint y, GLsizei w, GLsizei h) { ctx->viewport[0] = x; ctx->viewport[1] = y; ctx->viewport[2] = w; ctx->viewport[3] = h; }
void ClearColor(GLfloat r, GLfloat g, GLfloat b, GLfloat a) { ctx->clear_color[0] = r; ctx->clear_color[1] = g; ctx->clear_color[2] = b; ctx->clear_color[3] = a; }
void ClearDepth(GLdouble depth) { ctx->clear_depth = depth; }

// ---- clears (gl.cc:2370-2518) -------------------------------------------------------------------
void Clear(GLbitfield mask) {
  const int* rect = ctx->scissor_test ? ctx->scissor : nullptr;
  float depth = (float)ctx->clear_depth;
  const bool want_depth = (mask & GL_DEPTH_BUFFER_BIT) && ctx->depth_mask;
  clear_rect(ctx->draw_fbo, rect, (mask & GL_COLOR_BUFFER_BIT) ? ctx->clear_color : nullptr, want_depth ? &depth : nullptr);
}
void ClearColorRect(GLuint fbo, GLint x, GLint y, GLsizei w, GLsizei h, GLfloat r, GLfloat g, GLfloat b, GLfloat a) {
  int rect[4] = {x, y, w, h};
  float color[4] = {r, g, b, a};
  clear_rect(fbo, rect, color, nullptr);
}
void ClearTexSubImage(GLenum, GLint, GLint, GLint, GLint, GLsizei, GLsizei, GLsizei, GLenum, GLenum, const void*) {
  set_error(GL_INVALID_OPERATION);  // not issued on this path (Device clears through framebuffers)
}
void ClearTexImage(GLenum, GLint, GLenum, GLenum, const void*) { set_error(GL_INVALID_OPERATION); }

// ---- the draw call (gl.cc:2702-2800 → draw_elements → draw_quad) -------------------------------
void DrawElementsInstanced(GLenum mode, GLsizei count, GLenum type, GLintptr, GLsizei instancecount) {
  if (instancecount <= 0) return;
  if (mode != GL_TRIANGLES || count != 6 || type != GL_UNSIGNED_SHORT || !ctx->cur_prog) { set_error(GL_INVALID_OPERATION); return; }
  Prog& p = ctx->prog[ctx->cur_prog];
  if (!p.linked) { set_error(GL_INVALID_OPERATION); return; }
  // the per-instance attributes: one interleaved buffer holding the kind's #[repr(C)] records
  Vao& v = cur_vao();
  GLuint ibuf = 0;
  int stride = 0;
  size_t first = ~(size_t)0;
  for (int i = 0; i < 16; i++) {
    const Attr& a = v.a[i];
    if (!a.enabled || a.divisor != 1) continue;
    if (ibuf && a.buf != ibuf) { set_error(GL_INVALID_OPERATION); return; }
    ibuf = a.buf;
    stride = a.stride;
    if (a.offset < first) first = a.offset;
  }
  if (!ibuf || stride <= 0) { set_error(GL_INVALID_OPERATION); return; }
  Buf& ib = ctx->buf[ibuf];
  // every fetched attribute must lie inside the buffer; the last record may be shorter than the stride,
  // in which case the records are repacked (the backend copies stride * n bytes)
  size_t rec_end = 0;
  for (int i = 0; i < 16; i++) {
    const Attr& a = v.a[i];
    if (!a.enabled || a.divisor != 1) continue;
    const size_t tb = (a.type == GL_UNSIGNED_BYTE || a.type == GL_BYTE) ? 1 : (a.type == GL_UNSIGNED_SHORT || a.type == GL_SHORT) ? 2 : 4;
    rec_end = std::max(rec_end, a.offset - first + (size_t)a.size * tb);
  }
  if (rec_end > (size_t)stride ||
      first + (size_t)stride * (size_t)(instancecount - 1) + rec_end > ib.data.size()) { set_error(GL_INVALID_OPERATION); return; }
  const uint8_t* inst_ptr = ib.data.data() + first;
  std::vector<uint8_t> padded;
  if (first + (size_t)stride * (size_t)instancecount > ib.data.size()) {
    padded.assign((size_t)stride * (size_t)instancecount, 0);
    memcpy(padded.data(), inst_ptr, ib.data.size() - first);
    inst_ptr = padded.data();
  }
  // SWGL implements LEQUAL and LESS only (gl.cc:1352-1361 asserts on anything else); the renderer's
  // batches use LEQUAL (renderer/mod.rs:2829).  Anything else is refused rather than drawn as LEQUAL.
  if (ctx->depth_test && ctx->depth_func != GL_LEQUAL) { set_error(GL_INVALID_ENUM); return; }
  if (!sync_tables()) return;
  if (!bind_target(ctx->draw_fbo, p.uTransform)) return;
  wrcu_draw_state st;
  memset(&st, 0, sizeof st);
  const int key = blend_key();
  if (key < 0) { set_error(GL_INVALID_OPERATION); return; }
  st.blend = key;
  Tex* color = nullptr;
  wrcu_tex depth = 0;
  fbo_attachments(ctx->draw_fbo, &color, &depth);
  st.depth = (ctx->depth_test && depth) ? (ctx->depth_mask ? WRCU_DEPTH_TEST_WRITE : WRCU_DEPTH_TEST) : WRCU_DEPTH_OFF;
  for (int i = 0; i < 3; i++) {
    Tex* t = tex_of(ctx->unit_tex[p.slot[i] & 15]);
    st.color[i] = t ? t->dev : 0;
  }
  if (Tex* m = tex_of(ctx->unit_tex[p.slot[9] & 15])) st.clip_mask = m->dev;
  st.scissor_enabled = ctx->scissor_test ? 1 : 0;
  memcpy(st.scissor, ctx->scissor, sizeof st.scissor);
  memcpy(st.blend_color, ctx->blend_color, sizeof st.blend_color);
  check(wrcu_draw_batch(ctx->dev, p.kind, p.feats, &st, inst_ptr, (size_t)stride, instancecount));
}

// ---- readback and copies --------------------------------------------------------------------------
void ReadPixels(GLint x, GLint y, GLsizei width, GLsizei height, GLenum format, GLenum, void* data) {
  Tex* color = nullptr;
  wrcu_tex depth = 0;
  if (!fbo_attachments(ctx->read_fbo, &color, &depth)) { set_error(GL_INVALID_OPERATION); return; }
  uint8_t* dst = (uint8_t*)data;
  const int bpp = bytes_per_pixel(color->ifmt);
  const size_t stride = (size_t)(ctx->pack_row_length > 0 ? ctx->pack_row_length : width) * bpp;
  if (width <= 0 || height <= 0) { set_error(GL_INVALID_VALUE); return; }
  if (ctx->pack_buffer) {
    Buf& b = ctx->buf[ctx->pack_buffer];
    const size_t off = (size_t)(uintptr_t)data, need = (size_t)(height - 1) * stride + (size_t)width * bpp;
    if (off > b.data.size() || off + need > b.data.size()) { set_error(GL_INVALID_OPERATION); return; }
    dst = b.data.data() + off;
  }
  check(wrcu_read_pixels(ctx->dev, color->dev, x, y, width, height, dst, stride));
  if (bpp == 4 && format == GL_RGBA)
    for (int r = 0; r < height; r++) {
      uint8_t* p = dst + (size_t)r * stride;
      for (int i = 0; i < width; i++) { uint8_t t = p[4 * i]; p[4 * i] = p[4 * i + 2]; p[4 * i + 2] = t; }
    }
}
static void copy_tex(Tex* s, Tex* d, int sx, int sy, int w, int h, int dx, int dy) {
  if (!s || !d || !s->dev || !d->dev) { set_error(GL_INVALID_OPERATION); return; }
  const int32_t r[4] = {sx, sy, w, h};
  check(wrcu_texture_copy(ctx->dev, s->dev, d->dev, r, dx, dy));
}
void BlitFramebuffer(GLint sx0, GLint sy0, GLint sx1, GLint sy1, GLint dx0, GLint dy0, GLint dx1, GLint dy1, GLbitfield mask,
                     GLenum) {
  if (!(mask & GL_COLOR_BUFFER_BIT)) return;
  if (sx1 - sx0 != dx1 - dx0 || sy1 - sy0 != dy1 - dy0 || sx1 <= sx0 || sy1 <= sy0) { set_error(GL_INVALID_OPERATION); return; }
  Tex *s = nullptr, *d = nullptr;
  wrcu_tex z = 0;
  if (!fbo_attachments(ctx->read_fbo, &s, &z) || !fbo_attachments(ctx->draw_fbo, &d, &z)) { set_error(GL_INVALID_OPERATION); return; }
  copy_tex(s, d, sx0, sy0, sx1 - sx0, sy1 - sy0, dx0, dy0);
}
void CopyImageSubData(GLuint src_name, GLenum, GLint, GLint sx, GLint sy, GLint, GLuint dst_name, GLenum, GLint, GLint dx, GLint dy,
                      GLint, GLsizei w, GLsizei h, GLsizei) {
  copy_tex(tex_of(src_name), tex_of(dst_name), sx, sy, w, h, dx, dy);
}
void CopyTexSubImage2D(GLenum, GLint, GLint xoffset, GLint yoffset, GLint x, GLint y, GLsizei w, GLsizei h) {
  Tex* s = nullptr;
  wrcu_tex z = 0;
  if (!fbo_attachments(ctx->read_fbo, &s, &z)) { set_error(GL_INVALID_OPERATION); return; }
  copy_tex(s, tex_of(ctx->unit_tex[ctx->active_unit]), x, y, w, h, xoffset, yoffset);
}

// ---- timer queries (EXT_timer_query, used by the GPU profiler only) ------------------------------
void BeginQuery(GLenum, GLuint) {}
void EndQuery(GLenum) {}
void GetQueryObjectui64v(GLuint, GLenum pname, GLuint64* params) { params[0] = pname == GL_QUERY_RESULT_AVAILABLE ? 1 : 0; }

// ---- software-compositor hooks (swgl/src/composite.h:485-590; compositor/sw_compositor.rs) --------------
// A locked resource is a texture pinned for the compositor: Composite() blits between two of them on the
// device (wrcu_composite_blit); GetResourceBuffer() hands out a host copy of the pixels (the reference
// returns its own CPU buffer) — read back at that moment, valid until the resource is unlocked.
struct Locked {
  GLuint tex = 0;
  int locks = 0;
  std::vector<uint8_t> host;
};
static std::map<GLuint, Locked*> g_locked;
static Locked* lock_tex(GLuint id) {
  Tex* t = tex_of(id);
  if (!t || !t->dev) { set_error(GL_INVALID_OPERATION); return nullptr; }
  Locked*& l = g_locked[id];
  if (!l) { l = new Locked(); l->tex = id; }
  l->locks++;
  return l;
}
void* LockTexture(GLuint tex) { return lock_tex(tex); }
void* LockFramebuffer(GLuint fbo) {
  auto it = ctx->fbo.find(fbo);
  if (it == ctx->fbo.end() || !it->second.color) { set_error(GL_INVALID_OPERATION); return nullptr; }
  return lock_tex(it->second.color);
}
void LockResource(void* r) { if (r) ((Locked*)r)->locks++; }
void UnlockResource(void* r) {
  if (!r) return;
  Locked* l = (Locked*)r;
  if (--l->locks <= 0) { l->locks = 0; std::vector<uint8_t>().swap(l->host); }
}
void* GetResourceBuffer(void* r, int32_t* w, int32_t* h, int32_t* stride) {
  Locked* l = (Locked*)r;
  Tex* t = l ? tex_of(l->tex) : nullptr;
  if (w) *w = t ? t->w : 0;
  if (h) *h = t ? t->h : 0;
  if (stride) *stride = t ? t->w * bytes_per_pixel(t->ifmt) : 0;
  if (!t) return nullptr;
  const size_t row = (size_t)t->w * bytes_per_pixel(t->ifmt);
  l->host.resize(row * t->h);
  if (wrcu_read_pixels(ctx->dev, t->dev, 0, 0, t->w, t->h, l->host.data(), row) != WRCU_OK) { set_error(GL_INVALID_OPERATION); return nullptr; }
  return l->host.data();
}
void Composite(void* dst, void* src, GLint sx, GLint sy, GLsizei sw, GLsizei sh, GLint dx, GLint dy, GLsizei dw, GLsizei dh,
               GLboolean opaque, GLboolean flipX, GLboolean flipY, GLenum filter, GLint cx, GLint cy, GLsizei cw, GLsizei ch) {
  if (!dst || !src) return;
  Tex *d = tex_of(((Locked*)dst)->tex), *s = tex_of(((Locked*)src)->tex);
  if (!d || !s || bytes_per_pixel(d->ifmt) != 4 || bytes_per_pixel(s->ifmt) != 4 || !d->dev || !s->dev) { set_error(GL_INVALID_OPERATION); return; }
  const int32_t sr[4] = {sx, sy, sw, sh}, dr[4] = {dx, dy, dw, dh}, cr[4] = {cx, cy, cw, ch};
  check(wrcu_composite_blit(ctx->dev, d->dev, s->dev, sr, dr, opaque ? 1 : 0, flipX ? 1 : 0, flipY ? 1 : 0,
                            filter == GL_LINEAR ? 1 : 0, cr));
}
void CompositeYUV(void* dst, void* y, void* u, void* v, int colorSpace, GLuint colorDepth, GLint sx, GLint sy, GLsizei sw, GLsizei sh,
                  GLint dx, GLint dy, GLsizei dw, GLsizei dh, GLboolean flipX, GLboolean flipY, GLint cx, GLint cy, GLsizei cw,
                  GLsizei ch) {
  if (!dst || !y || !u || !v) return;  // (composite.h:1342-1344)
  Tex *d = tex_of(((Locked*)dst)->tex), *ty = tex_of(((Locked*)y)->tex), *tu = tex_of(((Locked*)u)->tex), *tv = tex_of(((Locked*)v)->tex);
  if (!d || !ty || !tu || !tv || !d->dev || !ty->dev || !tu->dev || !tv->dev || bytes_per_pixel(d->ifmt) != 4) { set_error(GL_INVALID_OPERATION); return; }
  const int32_t sr[4] = {sx, sy, sw, sh}, dr[4] = {dx, dy, dw, dh}, cr[4] = {cx, cy, cw, ch};
  check(wrcu_composite_blit_yuv(ctx->dev, d->dev, ty->dev, tu->dev, tv->dev, colorSpace, colorDepth, sr, dr, flipX ? 1 : 0,
                                flipY ? 1 : 0, cr));
}

}  // extern "C"
