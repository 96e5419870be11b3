// blit_yuv.cuh — CompositeYUV of the SWGL surface (swgl/src/composite.h:1335-1384): Gecko's SwCompositor
// converting a video frame (three 8-bit planes, chroma at full or half resolution) into a BGRA destination
// while scaling it.  linear_convert_yuv (composite.h:1146-1205) walks rows; linear_row_yuv (993-1144)
// walks a row in 4-pixel chunks on INTEGER coordinates (15 fractional bits), in three phases:
//   chunks whose first sample lies left of the planes      textureLinearRowR8 / textureLinearRowPairedR8
//   chunks that stay 4 texels inside both planes           upscaleYUV42R8 (half-resolution chroma path)
//   the rest, and a partial last chunk                     textureLinearRowR8 / textureLinearRowPairedR8
// Every quantity of chunk n is a closed form of n (the coordinates advance by integer additions), so a
// THREAD takes a (row, chunk) and reproduces the reference's lanes for it; the host computes the
// row-invariant start lanes and the phase boundaries with the reference's own float and integer steps.
// 10-, 12- and 16-bit planes (R16 textures, colorDepth > 8) take one phase: every chunk goes through
// textureLinearUnpackedR16 >> (colorDepth - 1 - 8) (composite.h:1025-1058), with the same 8-bit matrix.
#pragma once
#include "shader_composite_yuv.cuh"

#define WR_YUV_STEP_BITS 8  // composite.h:863
struct YuvBlitArgs {
  uint8_t* dst; int dst_pitch;
  int dx, dy;            // destination pixel of (row 0, chunk 0)
  int span, rows;        // dstBounds width / height
  const uint8_t *yp, *up, *vp;
  int y_pitch, c_pitch, yw, yh, cw, ch;
  int yU0[4], cU0[4];    // cast(init_interp(srcUV.x, srcDU) * (1 << STEP_BITS)), and the chroma lanes
  int yDU, cDU;          // per-chunk steps
  float v0, dv, cv0, cdv;  // quantised row coordinates: srcUV.y, srcDUV.y, chromaUV.y, chromaDUV.y
  int fast;              // the half-resolution fast path's condition holds
  int pre, inside;       // chunks before the upscale phase, pixels inside it
  int color_space;       // YUVRangedColorSpace (composite.h:1210-1218): same numbering as yuv.glsl's
  int rescale_bits;      // R16 planes: colorDepth - 1 - 8
};

WRD int wr_yb_clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
// one lane of textureLinearRowR8 (composite.h:796-817): ixq has 7 fractional bits
WRD int wr_yb_row_sample(const uint8_t* row0, int stride_v, int frac_v, int width, int ixq) {
  int ix = ixq >> 7;
  const int fracx = ((ix >= 0 ? ixq : 0) | (ix > width - 2 ? -1 : 0)) & 0x7F;
  ix = wr_yb_clamp(ix, 0, width - 2);  // clampCoord(ix, width - 1)
  const uint8_t* row1 = row0 + stride_v;
  const int t0 = row0[ix], t1 = row0[ix + 1], b0 = row1[ix], b1 = row1[ix + 1];
  const int l = t0 + (((b0 - t0) * frac_v) >> 7), h = t1 + (((b1 - t1) * frac_v) >> 7);
  return l + (((h - l) * fracx) >> 7);
}
WRD int wr_yb_vlerp(const uint8_t* row0, int stride_v, int frac_v, int i) {  // ycSrc0 + (((ycSrc1 - ycSrc0) * ycFracV) >> 7)
  const int a = row0[i], b = row0[i + stride_v];
  return a + (((b - a) * frac_v) >> 7);
}
WRD uint32_t wr_yb_pack(const Px& p) { return (uint32_t)p.b | ((uint32_t)p.g << 8) | ((uint32_t)p.r << 16) | 0xFF000000u; }

// get_ycbcr_info + YUVMatrix::From (composite.h:1296-1318, 664-741): SWGL always does 8-bit math here
WRD YuvFixed wr_yuv_blit_matrix(int color_space) {
  float bias[3], m[9];
  wr_yuv_color_matrix(color_space, 3, 8, bias, m);
  return wr_yuv_fixed_from(bias, m, 0);
}

// chunk n of row r: up to four BGRA pixels
WRD void wr_yuv_blit_chunk(const YuvBlitArgs& a, const YuvFixed& fm, int r, int n) {
  int yV = (int)wr_repeat_add(a.v0, a.dv, r), cV = (int)wr_repeat_add(a.cv0, a.cdv, r);
  const int yFracV = yV & 0x7F, cFracV = cV & 0x7F;
  yV >>= 7;
  cV >>= 7;
  const uint8_t* yRow = a.yp + (size_t)wr_yb_clamp(yV, 0, a.yh - 1) * a.y_pitch;
  const int yStrideV = (yV >= 0 && yV < a.yh - 1) ? a.y_pitch : 0;
  const size_t cOff = (size_t)wr_yb_clamp(cV, 0, a.ch - 1) * a.c_pitch;
  const uint8_t *uRow = a.up + cOff, *vRow = a.vp + cOff;
  const int cStrideV = (cV >= 0 && cV < a.ch - 1) ? a.c_pitch : 0;
  int Y[4], U[4], V[4];
  const int m = n - a.pre;
  if (a.fast && m >= 0 && 4 * m < a.inside) {
    // ---- upscaleYUV42R8 (composite.h:869-986), iteration m ----
    int yI[4], yIn[4], yfx[4];
    for (int j = 0; j < 4; j++) {
      const int u0 = a.yU0[j] + a.pre * a.yDU + m * a.yDU;
      yI[j] = u0 >> (WR_YUV_STEP_BITS + 7);
      yIn[j] = (u0 + a.yDU) >> (WR_YUV_STEP_BITS + 7);
      yfx[j] = (u0 >> WR_YUV_STEP_BITS) & 0x7F;  // (ycFracX >> 9): the coordinate's 7-bit fraction
    }
    // chroma coordinates: the averages of lanes (0,1) and (2,3) — taps 0.5 and 1.5 of the chunk
    int cs[4];
    for (int j = 0; j < 4; j++) cs[j] = a.cU0[j] + a.pre * a.cDU;
    const int ca = ((cs[0] + cs[1]) >> 1) + m * a.cDU, cb = ((cs[2] + cs[3]) >> 1) + m * a.cDU;
    const int cI0 = ca >> (WR_YUV_STEP_BITS + 7), cI1 = cb >> (WR_YUV_STEP_BITS + 7);
    const int cIn0 = (ca + a.cDU) >> (WR_YUV_STEP_BITS + 7);
    const int cfx0 = (ca >> WR_YUV_STEP_BITS) & 0x7F, cfx1 = (cb >> WR_YUV_STEP_BITS) & 0x7F;
    // current and next combined samples (rows blended)
    int ys[4], ysn[2], us[2], vs[2], usn[2], vsn[2];
    for (int j = 0; j < 4; j++) ys[j] = wr_yb_vlerp(yRow, yStrideV, yFracV, yI[0] + j);
    for (int j = 0; j < 2; j++) {
      ysn[j] = wr_yb_vlerp(yRow, yStrideV, yFracV, yIn[0] + j);
      us[j] = wr_yb_vlerp(uRow, cStrideV, cFracV, cI0 + j);
      vs[j] = wr_yb_vlerp(vRow, cStrideV, cFracV, cI0 + j);
      usn[j] = wr_yb_vlerp(uRow, cStrideV, cFracV, cIn0 + j);
      vsn[j] = wr_yb_vlerp(vRow, cStrideV, cFracV, cIn0 + j);
    }
    // the Y shuffles: yshuf = current samples, yshufn = their right neighbours
    int sh[4] = {ys[0], ys[1], ys[2], ys[3]};
    int shn[4] = {ys[1], ys[2], ys[3], yIn[0] == yI[3] ? ysn[1] : ysn[0]};
    if (yI[1] == yI[0]) { sh[3] = sh[2]; sh[2] = sh[1]; sh[1] = sh[0]; shn[3] = shn[2]; shn[2] = shn[1]; shn[1] = shn[0]; }  // .xxyz
    if (yI[2] == yI[1]) { sh[3] = sh[2]; sh[2] = sh[1]; shn[3] = shn[2]; shn[2] = shn[1]; }                                  // .xyyz
    if (yI[3] == yI[2]) { sh[3] = sh[2]; shn[3] = shn[2]; }                                                                  // .xyzz
    // chroma: [u0, u1, v0, v1] and neighbours [u1, next, v1, next]
    int cu[2] = {us[0], us[1]}, cv[2] = {vs[0], vs[1]};
    int cun[2] = {us[1], cIn0 == cI1 ? usn[1] : usn[0]}, cvn[2] = {vs[1], cIn0 == cI1 ? vsn[1] : vsn[0]};
    if (cI1 == cI0) { cu[1] = cu[0]; cv[1] = cv[0]; cun[1] = cun[0]; cvn[1] = cvn[0]; }  // .xxzz
    for (int j = 0; j < 4; j++) Y[j] = sh[j] + (((shn[j] - sh[j]) * yfx[j]) >> 7);
    const int uA = cu[0] + (((cun[0] - cu[0]) * cfx0) >> 7), uB = cu[1] + (((cun[1] - cu[1]) * cfx1) >> 7);
    const int vA = cv[0] + (((cvn[0] - cv[0]) * cfx0) >> 7), vB = cv[1] + (((cvn[1] - cv[1]) * cfx1) >> 7);
    // samples 0.25, 0.75, 1.25, 1.75 from the taps at 0.5 and 1.5
    U[0] = uA + ((uA - uB) >> 2); U[1] = uA + ((uB - uA) >> 2); U[2] = uB + ((uA - uB) >> 2); U[3] = uB + ((uB - uA) >> 2);
    V[0] = vA + ((vA - vB) >> 2); V[1] = vA + ((vB - vA) >> 2); V[2] = vB + ((vA - vB) >> 2); V[3] = vB + ((vB - vA) >> 2);
  } else {
    for (int j = 0; j < 4; j++) {
      const int yq = (a.yU0[j] + n * a.yDU) >> WR_YUV_STEP_BITS, cq = (a.cU0[j] + n * a.cDU) >> WR_YUV_STEP_BITS;
      Y[j] = wr_yb_row_sample(yRow, yStrideV, yFracV, a.yw, yq);
      U[j] = wr_yb_row_sample(uRow, cStrideV, cFracV, a.cw, cq);
      V[j] = wr_yb_row_sample(vRow, cStrideV, cFracV, a.cw, cq);
    }
  }
  uint32_t* d = (uint32_t*)(a.dst + (size_t)(a.dy + r) * a.dst_pitch) + a.dx + 4 * n;
  const int cnt = min(4, a.span - 4 * n);
  for (int j = 0; j < cnt; j++) d[j] = wr_yb_pack(wr_yuv_convert(fm, Y[j], U[j], V[j]));
}

// chunk n of row r, R16 planes (linear_row_yuv's R16 branch, composite.h:1025-1058)
WRD void wr_yuv_blit_chunk16(const YuvBlitArgs& a, const YuvFixed& fm, int r, int n) {
  const int yV = (int)wr_repeat_add(a.v0, a.dv, r), cV = (int)wr_repeat_add(a.cv0, a.cdv, r);
  uint32_t* d = (uint32_t*)(a.dst + (size_t)(a.dy + r) * a.dst_pitch) + a.dx + 4 * n;
  const int cnt = min(4, a.span - 4 * n);
  for (int j = 0; j < cnt; j++) {
    const int yq = (a.yU0[j] + n * a.yDU) >> WR_YUV_STEP_BITS, cq = (a.cU0[j] + n * a.cDU) >> WR_YUV_STEP_BITS;
    int Y, U, V;
    wr_texture_linear_16(a.yp, a.y_pitch, a.yw, a.yh, 1, yq, yV, &Y);
    wr_texture_linear_16(a.up, a.c_pitch, a.cw, a.ch, 1, cq, cV, &U);
    wr_texture_linear_16(a.vp, a.c_pitch, a.cw, a.ch, 1, cq, cV, &V);
    d[j] = wr_yb_pack(wr_yuv_convert(fm, Y >> a.rescale_bits, U >> a.rescale_bits, V >> a.rescale_bits));
  }
}

#ifdef WRCU_HOSTEMU
static void wr_sw_composite_blit_yuv(YuvBlitArgs a) {
  const YuvFixed fm = wr_yuv_blit_matrix(a.color_space);
  for (int r = 0; r < a.rows; r++)
    for (int n = 0; 4 * n < a.span; n++) wr_yuv_blit_chunk(a, fm, r, n);
}
static void wr_sw_composite_blit_yuv16(YuvBlitArgs a) {
  const YuvFixed fm = wr_yuv_blit_matrix(a.color_space);
  for (int r = 0; r < a.rows; r++)
    for (int n = 0; 4 * n < a.span; n++) wr_yuv_blit_chunk16(a, fm, r, n);
}
#else
__global__ void wr_sw_composite_blit_yuv(YuvBlitArgs a) {
  __shared__ YuvFixed fm;
  if (threadIdx.x == 0 && threadIdx.y == 0) fm = wr_yuv_blit_matrix(a.color_space);
  __syncthreads();
  const int n = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
  if (4 * n < a.span && r < a.rows) wr_yuv_blit_chunk(a, fm, r, n);
}
__global__ void wr_sw_composite_blit_yuv16(YuvBlitArgs a) {
  __shared__ YuvFixed fm;
  if (threadIdx.x == 0 && threadIdx.y == 0) fm = wr_yuv_blit_matrix(a.color_space);
  __syncthreads();
  const int n = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
  if (4 * n < a.span && r < a.rows) wr_yuv_blit_chunk16(a, fm, r, n);
}
#endif
