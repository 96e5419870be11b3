// shader_composite_yuv.cuh — composite with WR_FEATURE_YUV (webrender/res/composite.glsl:14-33,
// 83-130, 163-176, 197-214 + webrender/res/yuv.glsl): external video surfaces converted
// YCbCr → RGB while they are composited.  8-bit planes: PLANAR (three R8 textures), NV12
// (R8 + RG8 or RGBA8) and INTERLEAVED (one BGRA texture); 10-, 12- and 16-bit planes: PLANAR (three
// R16 textures) and NV12 / P010 (R16 + RG16), LSB-aligned except P010 (see wr_yuv_rescale).
//
// Span body (len & ~3): swgl_commitTextureLinearYUV → blendYUV → blendYUVFallback
// (swgl/src/swgl_ext.h:1006-1187): every plane is sampled through the fallback bilinear filter
// on its own quantised uv running sum, and the three samples go through the 6/7-bit fixed-point
// YUVMatrix of swgl/src/composite.h:636-779.  It only runs when every plane's sampler is
// LINEAR; otherwise — and for the len & 3 tail — the fragment shader's float matrix
// (sample_yuv, yuv.glsl:183-246) is used.
#pragma once
#include "raster.cuh"
#include "setup_common.cuh"
#include "setup_brush.cuh"
#include "texspan.cuh"

// textureLinearPlanarRG8 for one lane (texture.h:589-638)
WRD void wr_texture_linear_rg8(const TexView& t, int ix, int iy, int* out) {
  int x = ix >> 7, y = iy >> 7;
  int cx = wr_clamp_coord(x, t.w - 1);
  int cy = wr_clamp_coord(y, t.h);
  const uint8_t* row0 = t.ptr + (size_t)cy * t.pitch + (size_t)cx * 2;
  const uint8_t* row1 = row0 + ((y >= 0 && y < t.h - 1) ? t.pitch : 0);
  int overread = x > t.w - 2 ? -1 : 0;
  int fx = (int)(short)((((ix & (x >= 0 ? -1 : 0)) | overread) & 0x7F) - overread);
  int fy = iy & 0x7F;
  for (int ch = 0; ch < 2; ch++) {
    int a0 = __ldg(row0 + ch), a1 = __ldg(row1 + ch), b0 = __ldg(row0 + 2 + ch), b1 = __ldg(row1 + 2 + ch);
    out[ch] = wr_lerp7(wr_lerp7(a0, a1, fy), wr_lerp7(b0, b1, fy), fx) & 0xFFFF;
  }
}

// a + (((b - a) * f) >> 16) << 1 in int16 lanes: the 15-bit lerp of the R16 / RG16 fetches in the generic
// (non-SSE) build (texture.h:680-700); f is the 7-bit fraction shifted left by 8
WRD int wr_lerp15(int a, int b, int f) {
  const int d = (int)(short)(b - a);
  return (int)(short)(a + (int)(short)((int)(short)((d * f) >> 16) << 1));
}
// textureLinearUnpackedR16 / textureLinearUnpackedRG16 for one lane (texture.h:650-830): `nch` 16-bit channels
// per texel, each shifted right by one into a signed 15-bit sample.  The x fraction is computed inline, not by
// computeFracX: past the last column pair it is 127/128, not 128/128.
WRD void wr_texture_linear_16(const uint8_t* base, int pitch, int w, int h, int nch, int ix, int iy, int* out) {
  const int x = ix >> 7, y = iy >> 7;
  const int cx = wr_clamp_coord(x, w - 1), cy = wr_clamp_coord(y, h);
  const uint16_t* row0 = (const uint16_t*)(base + (size_t)cy * pitch) + (size_t)cx * nch;
  const uint16_t* row1 = (const uint16_t*)((const uint8_t*)row0 + ((y >= 0 && y < h - 1) ? pitch : 0));
  const int fx = (((ix & (x >= 0 ? -1 : 0)) | (x > w - 2 ? -1 : 0)) & 0x7F) << 8;
  const int fy = (iy & 0x7F) << 8;
  for (int ch = 0; ch < nch; ch++) {
    const int a0 = __ldg(row0 + ch) >> 1, a1 = __ldg(row1 + ch) >> 1;
    const int b0 = __ldg(row0 + nch + ch) >> 1, b1 = __ldg(row1 + nch + ch) >> 1;
    out[ch] = wr_lerp15(wr_lerp15(a0, a1, fy), wr_lerp15(b0, b1, fy), fx);
  }
}
WRD int wr_texture_linear_r16(const TexView& t, int ix, int iy) {
  int v;
  wr_texture_linear_16(t.ptr, t.pitch, t.w, t.h, 1, ix, iy, &v);
  return v;
}

// texture() of the fragment path for the plane formats (adds RG8 to wr_tex_fragment; HDR: R16 and RG16 only)
template <bool HDR>
WRD void wr_yuv_tex_fragment(const TexView& t, float cu, float cv, float* out) {
  if (HDR) {
    const int nch = t.fmt == WRCU_FMT_R16 ? 1 : 2;
    float s[2] = {0.0f, 0.0f};
    if (t.filter == WRCU_LINEAR) {
      // textureLinearR16 / textureLinearRG16 (texture.h:723-729, 823-830): int15 / 32767; RG16's red channel is
      // read back as the unsigned low half of its 32-bit lane
      int v[2];
      wr_texture_linear_16(t.ptr, t.pitch, t.w, t.h, nch, (int)wr_linear_quantize(cu, t.w), (int)wr_linear_quantize(cv, t.h), v);
      s[0] = (float)(nch == 2 ? (v[0] & 0xFFFF) : v[0]) * (1.0f / 32767.0f);
      if (nch == 2) s[1] = (float)v[1] * (1.0f / 32767.0f);
    } else {
      // texelFetchR16 / texelFetchRG16 (texture.h:149-176): u16 / 65535
      int x = wr_clamp_coord((int)(cu * (float)t.w), t.w), y = wr_clamp_coord((int)(cv * (float)t.h), t.h);
      const uint16_t* p = (const uint16_t*)(t.ptr + (size_t)y * t.pitch) + (size_t)x * nch;
      for (int ch = 0; ch < nch; ch++) s[ch] = (float)__ldg(p + ch) * (1.0f / 65535.0f);
    }
    out[0] = s[0];
    out[1] = s[1];
    out[2] = 0.0f;
    out[3] = 1.0f;
    return;
  }
  if (t.fmt != WRCU_FMT_RG8) {
    wr_tex_fragment(t, cu, cv, out);
    return;
  }
  int rg[2];
  if (t.filter == WRCU_LINEAR) {
    wr_texture_linear_rg8(t, (int)wr_linear_quantize(cu, t.w), (int)wr_linear_quantize(cv, t.h), rg);
  } else {
    int x = wr_clamp_coord((int)(cu * (float)t.w), t.w), y = wr_clamp_coord((int)(cv * (float)t.h), t.h);
    rg[0] = __ldg(t.ptr + (size_t)y * t.pitch + 2 * x);
    rg[1] = __ldg(t.ptr + (size_t)y * t.pitch + 2 * x + 1);
  }
  out[0] = (float)rg[0] * (1.0f / 255.0f);
  out[1] = (float)rg[1] * (1.0f / 255.0f);
  out[2] = 0.0f;
  out[3] = 1.0f;
}

// YUVMatrix (composite.h:636-741) in CmdCold::i-style ints
struct YuvFixed {
  int bu, rv, gu, gv, y_coeff, y_bias, uv_bias, br_y_mask;
};
WRD int wr_yuv_addsat(int x, int y) { return max(-32768, min(32767, x + y)); }  // composite.h:592-611
WRD int wr_yuv_pack8(int v) {  // genericPackWide (texture.h:13-21)
  unsigned p = (unsigned)v & 0xFFFFu;
  p = ((p | (p > 255u ? 0xFFFFu : 0u)) + (p >> 15)) & 0xFFFFu;
  return (int)(p & 0xFFu);
}
// YUVMatrix::convert (composite.h:743-778), one pixel
WRD Px wr_yuv_convert(const YuvFixed& m, int y, int u, int v) {
  int yy = (int)(short)((unsigned short)((unsigned)y * (unsigned)m.y_coeff) >> 1);
  yy = (int)(short)(yy - m.y_bias);
  int du = (int)(short)(u - m.uv_bias), dv = (int)(short)(v - m.uv_bias);
  int b = wr_yuv_addsat(yy & m.br_y_mask, (int)(short)(m.bu * du)) >> 6;
  int r = wr_yuv_addsat(yy & m.br_y_mask, (int)(short)(m.rv * dv)) >> 6;
  int g = wr_yuv_addsat(yy, wr_yuv_addsat((int)(short)(m.gu * du), (int)(short)(m.gv * dv))) >> 6;
  return Px{wr_yuv_pack8(b), wr_yuv_pack8(g), wr_yuv_pack8(r), 255};
}

// One shader, two kernels: HDR = false samples the 8-bit plane sets, HDR = true the 16-bit ones (R16 luma; the
// launch picks it from the luma plane's format), so the 8-bit kernel carries none of the 16-bit code.
// CmdCold: g[0..11] vUVBounds_y/u/v, g[12..14] vYcbcrBias, g[15..23] vRgbFromDebiasedYcbcr
// (column-major), g[24..31] YuvFixed (int bits), g[32] != 0: clamp rgb (brush_yuv_image ALPHA_PASS,
// yuv.glsl:239-243), g[33] (int bits) rescaleBits of 16-bit planes; i[0] = vYuvFormat.x, i[1] = planes,
// i[2..3] the u chain table
struct CompositeYuvShader {
  struct PlaneRow {
    float bu[4], bv[4];  // quantised uv lanes of chunk kb
    float ustep, vstep, minu, minv, maxu, maxv;
    int exact;  // bit 0: u sums exact (wr_sum_exact), bit 1: v sums
  };
  struct Row {
    float o[6], step[6];
    int body_len, kb, frag_accum;
    const float* chain;  // u running sums of every chunk of the span, from the setup kernel (see wr_yuv_chain_table)
    int nch;
    PlaneRow p[3];
  };
  WRD_MEMBER const TexView& plane(const RasterArgs& a, int p) {
    return p == 0 ? a.color0 : (p == 1 ? a.color1 : a.color2);
  }
  template <bool HDR>
  WRD_MEMBER void row_setup_t(const RasterArgs& a, const CmdHot& c, int y, int tx0, bool rgba, Row& r) {
    const CmdCold& k = a.cold[c.cold];
    wr_row_interp<6>(a, k, c, y, r.o, r.step);
    int len = c.x1 - c.x0;
    const int planes = k.i[1];
    bool ok = rgba && len >= 4;
    for (int p = 0; p < planes; p++) ok = ok && plane(a, p).filter == WRCU_LINEAR;
    // sampleYUV's format switches (swgl_ext.h:1009-1127)
    if (HDR) ok = ok && (planes == 3 ? a.color1.fmt == WRCU_FMT_R16 && a.color2.fmt == WRCU_FMT_R16
                                     : planes == 2 && a.color1.fmt == WRCU_FMT_RG16);
    else if (planes == 3) ok = ok && a.color0.fmt == WRCU_FMT_R8 && a.color1.fmt == WRCU_FMT_R8 && a.color2.fmt == WRCU_FMT_R8;
    else if (planes == 2) ok = ok && a.color0.fmt == WRCU_FMT_R8 && (a.color1.fmt == WRCU_FMT_RG8 || a.color1.fmt == WRCU_FMT_RGBA8);
    else ok = ok && a.color0.fmt == WRCU_FMT_RGBA8;
    r.body_len = ok ? (len & ~3) : 0;
    r.kb = max(0, (max(tx0, (int)c.x0) - (int)c.x0) >> 2);
    r.frag_accum = !r.body_len && len >= 4;
    if (!r.body_len && !r.frag_accum) return;
    // Start lanes and per-chunk steps of the six running sums (three planes x u,v).  Span body:
    // LINEAR_QUANTIZE_UV (swgl_ext.h:160-168) per plane.  No span shader (a NEAREST plane): the
    // fragment loop advances the varyings chunk by chunk (run() -> step_interp_inputs, vUV +=
    // interp_step) — scaled video samples exactly on texel boundaries, where that sum's rounding
    // decides the texel.
    float uvj[4][6];
    for (int j = 0; j < 4; j++) wr_interp_at<6>(a, r.o, r.step, j, uvj[j]);
    float q[3][2][4], st[3][2];
    for (int p = 0; p < 3; p++) {
      const TexView& t = plane(a, p);
      PlaneRow& pr = r.p[p];
      for (int ax = 0; ax < 2; ax++) {
        for (int j = 0; j < 4; j++)
          q[p][ax][j] = r.body_len ? wr_linear_quantize(uvj[j][2 * p + ax], ax ? t.h : t.w) : uvj[j][2 * p + ax];
        st[p][ax] = r.body_len ? 4.0f * (q[p][ax][1] - q[p][ax][0]) : __fmul_rn(r.step[2 * p + ax], 4.0f);
      }
      pr.ustep = st[p][0];
      pr.vstep = st[p][1];
      if (r.body_len) {
        const float* b = k.g + 4 * p;
        pr.minu = wr_max(wr_linear_quantize(b[0], t.w), 0.0f);
        pr.minv = wr_max(wr_linear_quantize(b[1], t.h), 0.0f);
        pr.maxu = wr_max(wr_linear_quantize(b[2], t.w), pr.minu);
        pr.maxv = wr_max(wr_linear_quantize(b[3], t.h), pr.minv);
      }
    }
    r.chain = nullptr;
    if (r.body_len && k.i[2] >= 0) {
      // The setup kernel walked the u sums of this surface once (they are the same on every row of an
      // axis-aligned surface, and v does not move along a row).  Valid for this row iff the row's
      // start lanes and steps are bit-identical to the ones the table was built from.
      const float* T = a.row_tab + k.i[2];
      bool same = true;
      for (int p = 0; p < planes; p++) {
        for (int j = 0; j < 4; j++) same = same && __float_as_uint(q[p][0][j]) == __float_as_uint(__ldg(T + p * 4 + j));
        same = same && __float_as_uint(st[p][0]) == __float_as_uint(__ldg(T + 12 + p)) && st[p][1] == 0.0f;
      }
      if (same) {
        r.chain = T + 16;
        r.nch = k.i[3];
        for (int p = 0; p < 3; p++) {
          for (int j = 0; j < 4; j++) { r.p[p].bu[j] = q[p][0][j]; r.p[p].bv[j] = q[p][1][j]; }
          r.p[p].exact = 0;
        }
        return;
      }
    }
#ifdef WRCU_HOSTEMU
    for (int p = 0; p < 3; p++) {
      wr_tex_seq_base(q[p][0], st[p][0], r.kb, r.p[p].bu);
      wr_tex_seq_base(q[p][1], st[p][1], r.kb, r.p[p].bv);
    }
#else
    {
      // 24 independent walks, the whole warp is here: lane l < 24 takes (plane, axis, chunk lane)
      // = (l >> 3, (l >> 2) & 1, l & 3); the results are broadcast (see wr_tex_bases)
      const int l = threadIdx.x & 31, lp = l >> 3, lax = (l >> 2) & 1, lj = l & 3;
      float x = 0.0f, sx = 0.0f;
#pragma unroll
      for (int p = 0; p < 3; p++)
#pragma unroll
        for (int ax = 0; ax < 2; ax++)
          if (lp == p && lax == ax) { x = wr_sel4(q[p][ax], lj); sx = st[p][ax]; }
      const float val = l < 24 ? wr_repeat_add(x, sx, r.kb) : 0.0f;
#pragma unroll
      for (int p = 0; p < 3; p++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          r.p[p].bu[j] = __shfl_sync(0xFFFFFFFFu, val, p * 8 + j);
          r.p[p].bv[j] = __shfl_sync(0xFFFFFFFFu, val, p * 8 + 4 + j);
        }
    }
#endif
    for (int p = 0; p < 3; p++)
      r.p[p].exact = (wr_sum_exact(r.p[p].bu, r.p[p].ustep) ? 1 : 0) | (wr_sum_exact(r.p[p].bv, r.p[p].vstep) ? 2 : 0);
  }
  template <bool HDR>
  WRD_MEMBER Px source_t(const RasterArgs& a, const CmdHot& c, const Row& r, int x) {
    const CmdCold& k = a.cold[c.cold];
    int rel = x - c.x0;
    const int planes = k.i[1], format = k.i[0];
    if (rel < r.body_len) {
      // blendYUVFallback (swgl_ext.h:1140-1157): uv += uv_step per chunk, clamp, sample, convert
      int j = rel & 3;
      int ii[3][2];
      for (int p = 0; p < planes; p++) {
        const PlaneRow& pr = r.p[p];
        const int m = (rel >> 2) - r.kb;
        float qu, qv;
        if (r.chain) {
          qu = __ldg(r.chain + (size_t)(p * 4 + j) * r.nch + (rel >> 2));
          qv = pr.bv[j];
        } else {
          qu = wr_sum_at(pr.bu[j], pr.ustep, m, pr.exact & 1);
          qv = wr_sum_at(pr.bv[j], pr.vstep, m, pr.exact & 2);
        }
        ii[p][0] = (int)wr_clamp(qu, pr.minu, pr.maxu);
        ii[p][1] = (int)wr_clamp(qv, pr.minv, pr.maxv);
      }
      int yv, uu, vv;
      if (HDR) {
        // 16-bit planes (swgl_ext.h:1078-1093, 1124-1140): 15-bit samples shifted down by rescaleBits
        const int rb = ((const int*)k.g)[33];
        yv = wr_texture_linear_r16(a.color0, ii[0][0], ii[0][1]) >> rb;
        if (planes == 3) {
          uu = wr_texture_linear_r16(a.color1, ii[1][0], ii[1][1]) >> rb;
          vv = wr_texture_linear_r16(a.color2, ii[2][0], ii[2][1]) >> rb;
        } else {
          int uv[2];
          wr_texture_linear_16(a.color1.ptr, a.color1.pitch, a.color1.w, a.color1.h, 2, ii[1][0], ii[1][1], uv);
          uu = uv[0] >> rb; vv = uv[1] >> rb;
        }
      } else if (planes == 3) {
        yv = wr_texture_linear_r8(a.color0, ii[0][0], ii[0][1]);
        uu = wr_texture_linear_r8(a.color1, ii[1][0], ii[1][1]);
        vv = wr_texture_linear_r8(a.color2, ii[2][0], ii[2][1]);
      } else if (planes == 2) {
        yv = wr_texture_linear_r8(a.color0, ii[0][0], ii[0][1]);
        if (a.color1.fmt == WRCU_FMT_RG8) {
          int rg[2];
          wr_texture_linear_rg8(a.color1, ii[1][0], ii[1][1], rg);
          uu = rg[0]; vv = rg[1];
        } else {  // RGBA8 chroma plane: u = lowHalf(ba) = byte 2, v = highHalf(rg) = byte 1
          Px c4 = wr_texture_linear_rgba8(a.color1, ii[1][0], ii[1][1]);
          uu = c4.r; vv = c4.g;
        }
      } else {  // interleaved: y = byte 1, u = byte 0, v = byte 2
        Px c4 = wr_texture_linear_rgba8(a.color0, ii[0][0], ii[0][1]);
        yv = c4.g; uu = c4.b; vv = c4.r;
      }
      YuvFixed m;
      const int* mi = (const int*)(k.g + 24);
      m.bu = mi[0]; m.rv = mi[1]; m.gu = mi[2]; m.gv = mi[3];
      m.y_coeff = mi[4]; m.y_bias = mi[5]; m.uv_bias = mi[6]; m.br_y_mask = mi[7];
      return wr_yuv_convert(m, yv, uu, vv);
    }
    // main() → sample_yuv (yuv.glsl:183-246)
    float uv[6];
    if (r.frag_accum) {
      int j = rel & 3;
      for (int p = 0; p < 3; p++) {
        const int m = (rel >> 2) - r.kb;
        float qu = wr_sum_at(r.p[p].bu[j], r.p[p].ustep, m, r.p[p].exact & 1);
        float qv = wr_sum_at(r.p[p].bv[j], r.p[p].vstep, m, r.p[p].exact & 2);
        uv[2 * p] = qu;
        uv[2 * p + 1] = qv;
      }
    } else {
      wr_interp_at<6>(a, r.o, r.step, rel, uv);
    }
    float cc[3][2];
    for (int p = 0; p < 3; p++) {
      cc[p][0] = wr_clamp(uv[2 * p], k.g[4 * p], k.g[4 * p + 2]);
      cc[p][1] = wr_clamp(uv[2 * p + 1], k.g[4 * p + 1], k.g[4 * p + 3]);
    }
    float s3[3] = {0.0f, 0.0f, 0.0f}, t4[4];
    if (format == 3) {
      wr_yuv_tex_fragment<HDR>(a.color0, cc[0][0], cc[0][1], t4); s3[0] = t4[0];
      wr_yuv_tex_fragment<HDR>(a.color1, cc[1][0], cc[1][1], t4); s3[1] = t4[0];
      wr_yuv_tex_fragment<HDR>(a.color2, cc[2][0], cc[2][1], t4); s3[2] = t4[0];
    } else if (format >= 0 && format <= 2) {
      wr_yuv_tex_fragment<HDR>(a.color0, cc[0][0], cc[0][1], t4); s3[0] = t4[0];
      wr_yuv_tex_fragment<HDR>(a.color1, cc[1][0], cc[1][1], t4); s3[1] = t4[0]; s3[2] = t4[1];
    } else if (format == 4) {
      wr_yuv_tex_fragment<HDR>(a.color0, cc[0][0], cc[0][1], t4); s3[0] = t4[1]; s3[1] = t4[2]; s3[2] = t4[0];
    }
    float dv[3] = {s3[0] - k.g[12], s3[1] - k.g[13], s3[2] - k.g[14]};
    float col[3];
    for (int q = 0; q < 3; q++)
      col[q] = __fadd_rn(__fadd_rn(__fmul_rn(k.g[15 + q], dv[0]), __fmul_rn(k.g[18 + q], dv[1])), __fmul_rn(k.g[21 + q], dv[2]));
    if (k.g[32] != 0.0f)
      for (int q = 0; q < 3; q++) col[q] = wr_clamp(col[q], 0.0f, 1.0f);
    Px o;
    o.r = wr_round_pixel(col[0], 255.0f) & 0xFFFF;
    o.g = wr_round_pixel(col[1], 255.0f) & 0xFFFF;
    o.b = wr_round_pixel(col[2], 255.0f) & 0xFFFF;
    o.a = 255;
    return o;
  }
  WRD_MEMBER void row_setup(const RasterArgs& a, const CmdHot& c, int y, int tx0, bool rgba, Row& r) {
    row_setup_t<false>(a, c, y, tx0, rgba, r);
  }
  WRD_MEMBER Px source(const RasterArgs& a, const CmdHot& c, const Row& r, int x, int, bool) { return source_t<false>(a, c, r, x); }
};
struct CompositeYuv16Shader : CompositeYuvShader {
  WRD_MEMBER void row_setup(const RasterArgs& a, const CmdHot& c, int y, int tx0, bool rgba, Row& r) {
    row_setup_t<true>(a, c, y, tx0, rgba, r);
  }
  WRD_MEMBER Px source(const RasterArgs& a, const CmdHot& c, const Row& r, int x, int, bool) { return source_t<true>(a, c, r, x); }
};

// get_yuv_color_info + get_rgb_from_ycbcr_info (yuv.glsl:79-161); m is column-major [col*3+row]
WRD void wr_yuv_color_matrix(int color_space, int format, int bit_depth, float* bias, float* m) {
  const float REC601[9] = {1.00000f, 1.00000f, 1.00000f, 0.00000f, -0.17207f, 0.88600f, 0.70100f, -0.35707f, 0.00000f};
  const float REC709[9] = {1.00000f, 1.00000f, 1.00000f, 0.00000f, -0.09366f, 0.92780f, 0.78740f, -0.23406f, 0.00000f};
  const float REC2020[9] = {1.00000f, 1.00000f, 1.00000f, 0.00000f, -0.08228f, 0.94070f, 0.73730f, -0.28568f, 0.00000f};
  const float GBR[9] = {0.0f, 1.0f, 0.0f, 0.0f, 0.0f, 1.0f, 1.0f, 0.0f, 0.0f};
  float channel_max = 255.0f;
  if (bit_depth > 8) channel_max = format == 1 ? (float)((1 << bit_depth) - 1) : 65535.0f;
  const int NARROW[4] = {16, 128, 235, 240};
  float narrow[4], zo[4];
  for (int q = 0; q < 4; q++) narrow[q] = (float)(NARROW[q] << (bit_depth - 8)) / channel_max;
  float all_ones = (float)((1 << bit_depth) - 1) / channel_max;
  const float* am;
  int range;  // 0 narrow, 1 full, 2 identity
  switch (color_space) {
    case 0: am = REC601; range = 0; break;
    case 1: am = REC601; range = 1; break;
    case 2: am = REC709; range = 0; break;
    case 3: am = REC709; range = 1; break;
    case 4: am = REC2020; range = 0; break;
    case 5: am = REC2020; range = 1; break;
    default: am = GBR; range = 2; break;
  }
  if (range == 0) { for (int q = 0; q < 4; q++) zo[q] = narrow[q]; }
  else if (range == 2) { zo[0] = 0.0f; zo[1] = 0.0f; zo[2] = all_ones; zo[3] = all_ones; }
  else { zo[0] = 0.0f; zo[1] = narrow[1]; zo[2] = all_ones; zo[3] = all_ones; }
  float scale[2] = {1.0f / (zo[2] - zo[0]), 1.0f / (zo[3] - zo[1])};
  bias[0] = zo[0]; bias[1] = zo[1]; bias[2] = zo[1];
  // rgb_from_yuv * diag(scale.x, scale.y, scale.y): mat3_scalar product (glsl.h:2418-2427)
  for (int cidx = 0; cidx < 3; cidx++) {
    float b[3] = {cidx == 0 ? scale[0] : 0.0f, cidx == 1 ? scale[1] : 0.0f, cidx == 2 ? scale[1] : 0.0f};
    for (int rr = 0; rr < 3; rr++)
      m[cidx * 3 + rr] = __fadd_rn(__fadd_rn(__fmul_rn(am[rr], b[0]), __fmul_rn(am[3 + rr], b[1])), __fmul_rn(am[6 + rr], b[2]));
  }
}

// YUVMatrix::From + constructor (composite.h:664-741)
WRD YuvFixed wr_yuv_fixed_from(const float* bias, const float* m, int rescale) {
  YuvFixed o;
  double y_coeff = (double)m[1];
  o.br_y_mask = m[0] == 0.0f ? 0 : -1;
  double gu = (double)m[3 + 1], bu = (double)m[3 + 2], rv = (double)m[6 + 0], gv = (double)m[6 + 1];
  double sc = (double)(1 << (6 - rescale));
  o.bu = (int)(short)(int)(bu * sc + 0.5);
  o.rv = (int)(short)(int)(rv * sc + 0.5);
  o.gu = -(int)(short)(int)(-gu * sc + 0.5);
  o.gv = -(int)(short)(int)(-gv * sc + 0.5);
  o.y_coeff = (int)(unsigned short)(int)(y_coeff * (double)(1 << (6 + 1 - rescale)) + 0.5);
  float bx255 = __fmul_rn(bias[0], 255.0f);
  o.y_bias = (int)(short)(int)((((double)bx255 * y_coeff) - 0.5) * 64.0);
  float by = __fmul_rn(bias[1], (float)(255 << rescale));
  o.uv_bias = (int)(short)(int)((double)by + 0.5);
  return o;
}

// The u running sums of a video surface, once per command instead of once per (row, tile).
// blendYUVFallback advances each plane's quantised uv by uv_step per 4-pixel chunk from the span
// start; a tile in the middle of a 4K-wide span needs the sum after up to 959 additions.  For an
// axis-aligned surface the start lanes and the step of u are the same on every row and v does not
// change along a row, so the whole u sequence — 12 chains (3 planes x 4 chunk lanes) x one value per
// chunk — is walked here with plain additions (the reference's own sequence) into the row-table
// pool.  Header: the 12 start lanes + 3 steps the table was built from; the raster kernel uses the
// table only on rows whose own start lanes and steps are bit-identical.
// One of the 24 half-chains of command idx: chain q = part % 12 (plane q / 4, chunk lane q % 4), half
// part / 12.  The second half starts from the exact sum at its first chunk (wr_repeat_add), then both
// proceed by plain additions.
WRD void wr_yuv_chain_fill(const SetupArgs& a, int idx, int part) {
  const CmdCold& k = a.cold[idx];
  float* T = a.row_tab + k.i[2];
  const int nch = k.i[3], q = part % 12, half = part / 12;
#ifdef WRCU_HOSTEMU
  const int m0 = 0, m1 = nch;
  if (half) return;
#else
  const int mid = nch >> 1;
  const int m0 = half ? mid : 0, m1 = half ? nch : mid;
#endif
  const float st = T[12 + (q >> 2)];
  float v = wr_repeat_add(T[q], st, m0);
  float* C = T + 16 + (size_t)q * nch;
  for (int m = m0; m < m1; m++) {
    C[m] = v;
    v = v + st;
  }
}

WRD void wr_yuv_chain_table(const SetupArgs& a, int idx, int planes, const TexView* const* tv) {
  const CmdHot h = a.hot[idx];
  CmdCold& k = a.cold[idx];
  if (!a.row_tab || (h.flags & CMD_GENERAL) || h.x1 <= h.x0) return;
  const int len = (int)h.x1 - (int)h.x0;
  if (len < 4) return;
  const int nch = (len >> 2) + 1;
  const int need = 16 + 12 * nch;
  const int off = atomicAdd(a.pool_ctr, need);
  if (off < 0 || off + need > a.row_cap) return;  // pool exhausted: the raster kernel walks the sums itself
  // the first row's interpolants, as wr_row_interp computes them (rows = 0)
  float o[6], step[6];
  {
    float y0c = (float)h.y0 + 0.5f;
    float dy = __fsub_rn(y0c, k.yt);
    float stepScale = __fdiv_rn(1.0f, __fsub_rn(k.xr, k.xl));
    if (!isfinite(stepScale)) stepScale = 0.0f;
    float x0f = __fsub_rn(__fadd_rn((float)h.x0, 0.5f), k.xl);
    for (int i = 0; i < 6; i++) {
      float sl = __fmul_rn(__fsub_rn(k.i_lb[i], k.i_lt[i]), k.yscale);
      float sr = __fmul_rn(__fsub_rn(k.i_rb[i], k.i_rt[i]), k.yscale);
      float li = __fadd_rn(k.i_lt[i], __fmul_rn(dy, sl));
      float ri = __fadd_rn(k.i_rt[i], __fmul_rn(dy, sr));
      float st = __fmul_rn(__fsub_rn(ri, li), stepScale);
      step[i] = st;
      o[i] = __fadd_rn(li, __fmul_rn(st, x0f));
    }
  }
  float* T = a.row_tab + off;
  float v[12], st[3];
  for (int j = 0; j < 4; j++) {
    float uv[6];
    wr_interp_at_plain<6>(o, step, j, uv);
    for (int p = 0; p < 3; p++) v[p * 4 + j] = p < planes ? wr_linear_quantize(uv[2 * p], tv[p]->w) : 0.0f;
  }
  for (int p = 0; p < 3; p++) st[p] = 4.0f * (v[p * 4 + 1] - v[p * 4 + 0]);
  for (int q = 0; q < 12; q++) T[q] = v[q];
  for (int p = 0; p < 3; p++) T[12 + p] = st[p];
  T[15] = 0.0f;
  k.i[2] = off;
  k.i[3] = nch;
#ifdef WRCU_HOSTEMU
  for (int q = 0; q < 12; q++) wr_yuv_chain_fill(a, idx, q);
#endif
}

// The plane sets the span and fragment stages sample (sampleYUV's format switches, swgl_ext.h:1009-1140):
// depth 8 keeps the 8-bit sets (no 16-bit plane, no P010); depth 10, 12 or 16 takes three R16 planes (PLANAR) or
// R16 + RG16 (NV12, P010).  Returns vRescaleFactor (composite.glsl:90-96: 16 - depth for the LSB-aligned formats,
// 0 for MSB-aligned P010), or -1 for any other combination.
WRD int wr_yuv_planes(int format) { return format == 3 ? 3 : (format == 0 || format == 1 ? 2 : (format == 4 ? 1 : 0)); }
WRD int wr_yuv_rescale(int format, int bit_depth, const TexView* const* tv) {
  if (bit_depth == 8) {
    if (format == 1) return -1;
    for (int p = 0; p < wr_yuv_planes(format); p++)
      if (tv[p]->fmt == WRCU_FMT_R16 || tv[p]->fmt == WRCU_FMT_RG16) return -1;
    return 0;
  }
  if (bit_depth != 10 && bit_depth != 12 && bit_depth != 16) return -1;
  if (format == 3) {
    if (tv[0]->fmt != WRCU_FMT_R16 || tv[1]->fmt != WRCU_FMT_R16 || tv[2]->fmt != WRCU_FMT_R16) return -1;
  } else if (format == 0 || format == 1) {
    if (tv[0]->fmt != WRCU_FMT_R16 || tv[1]->fmt != WRCU_FMT_RG16) return -1;
  } else {
    return -1;
  }
  return format == 1 ? 0 : 16 - bit_depth;
}

// An instance that is not drawn: an empty command with wr_emit_quad's cold record for a culled quad — the warp-wide
// row-table and chain fills after the vertex stage read every instance's record, which must not be a stale one.
WRD void wr_yuv_reject(const SetupArgs& a, int idx) {
  CmdHot h = CmdHot{};
  h.cold = idx;
  a.hot[idx] = h;
  CmdCold& k = a.cold[idx];
  k.row_off = -1;
  k.row_n = 0;
  k.fail_off = -1;
  k.i[2] = -1;
}

// composite vertex stage, YUV branch (composite.glsl:73-130)
WRD void wr_setup_composite_yuv_one(const SetupArgs& a, int idx) {
  const float* f = (const float*)(a.instances + (size_t)idx * a.stride);
  const float* dr = f;
  const float* cr = f + 4;
  float flipx = f[28], flipy = f[29];
  QuadOut q;
  memset(&q, 0, sizeof q);
  float rect[4] = {(dr[2] - dr[0]) * flipx + dr[0], (dr[3] - dr[1]) * flipy + dr[1],
                   (dr[0] - dr[2]) * flipx + dr[2], (dr[1] - dr[3]) * flipy + dr[3]};
  int color_space = (int)f[13], format = (int)f[14], bit_depth = (int)f[15];
  int planes = wr_yuv_planes(format);
  const TexView* tv[3] = {&a.color0, &a.color1, &a.color2};
  const int rescale = wr_yuv_rescale(format, bit_depth, tv);
  bool bad = rescale < 0 || planes == 0;
  for (int p = 0; p < planes; p++) bad = bad || !tv[p]->ptr;
  if (bad) {
    wr_yuv_reject(a, idx);
    atomicAdd(&a.info->unsupported, 1);
    atomicAdd(a.err_counter, 1);
    return;
  }
  const float ax[4] = {0.0f, 1.0f, 1.0f, 0.0f}, ay[4] = {0.0f, 0.0f, 1.0f, 1.0f};
  for (int kx = 0; kx < 4; kx++) {
    float wx = (rect[2] - rect[0]) * ax[kx] + rect[0], wy = (rect[3] - rect[1]) * ay[kx] + rect[1];
    float cx = wr_clamp(wx, cr[0], cr[2]), cy = wr_clamp(wy, cr[1], cr[3]);
    float ux = (cx - rect[0]) / (rect[2] - rect[0]), uy = (cy - rect[1]) / (rect[3] - rect[1]);
    for (int p = 0; p < planes; p++) {  // write_uv_rect (yuv.glsl:163-178)
      const float* uvr = f + 16 + 4 * p;
      q.interp[kx][2 * p] = ((uvr[2] - uvr[0]) * ux + uvr[0]) / (float)tv[p]->w;
      q.interp[kx][2 * p + 1] = ((uvr[3] - uvr[1]) * uy + uvr[1]) / (float)tv[p]->h;
    }
    q.pos[kx] = wr_mat_mul(a.tgt.proj, make_float4(cx, cy, 0.0f, 1.0f));
  }
  q.n_interp = 6;
  q.flags = CMD_TEXTURED;
  q.col[0] = q.col[1] = q.col[2] = q.col[3] = 255;
  int unsupported = 0;
  bool ok = wr_emit_quad(a, idx, q, &unsupported);
  if (ok) {
    CmdCold* k = &a.cold[idx];
    for (int p = 0; p < 3; p++) {
      const float* uvr = f + 16 + 4 * p;
      float tw = (float)tv[p]->w, th = (float)tv[p]->h;
      k->g[4 * p + 0] = (uvr[0] + 0.5f) / tw;
      k->g[4 * p + 1] = (uvr[1] + 0.5f) / th;
      k->g[4 * p + 2] = (uvr[2] - 0.5f) / tw;
      k->g[4 * p + 3] = (uvr[3] - 0.5f) / th;
    }
    wr_yuv_color_matrix(color_space, format, bit_depth, &k->g[12], &k->g[15]);
    YuvFixed m = wr_yuv_fixed_from(&k->g[12], &k->g[15], rescale);
    int* mi = (int*)(k->g + 24);
    mi[0] = m.bu; mi[1] = m.rv; mi[2] = m.gu; mi[3] = m.gv;
    mi[4] = m.y_coeff; mi[5] = m.y_bias; mi[6] = m.uv_bias; mi[7] = m.br_y_mask;
    mi[9] = (16 - rescale - 1) - 8;  // rescaleBits (swgl_ext.h:1087-1088)
    k->i[0] = format;
    k->i[1] = planes;
    k->i[2] = -1;
    k->i[3] = 0;
    k->g[32] = 0.0f;
    wr_yuv_chain_table(a, idx, planes, tv);
  }
  if (unsupported) {
    atomicAdd(&a.info->unsupported, 1);
    atomicAdd(a.err_counter, 1);
  }
}
// WR_SETUP_KERNEL plus the chain tables: after its 32 instances are emitted the warp fills the table of
// each in turn, 24 lanes on the 12 chains x 2 halves (a single thread would take ~70 us for a 4K span).
#ifdef WRCU_HOSTEMU
#define WR_SETUP_KERNEL_YUV(name) WR_SETUP_KERNEL(name)
#else
#define WR_SETUP_KERNEL_YUV(name)                                                              \
  __device__ __noinline__ void name##_block(const SetupArgs& a, int idx) {                     \
    if (idx == 0 && a.info_next) wr_reset_batch_info(a.info_next);                             \
    if (idx < a.n) name##_one(a, idx);                                                         \
    __syncwarp();                                                                              \
    wr_fill_row_tables_warp(a, idx);                                                           \
    const int lane = threadIdx.x & 31, wbase = idx - lane;                                     \
    const bool has = idx < a.n && a.hot[idx].x1 > a.hot[idx].x0 && a.cold[idx].i[2] >= 0;      \
    unsigned m = __ballot_sync(0xFFFFFFFFu, has);                                              \
    while (m) {                                                                                \
      const int src = __ffs((int)m) - 1;                                                       \
      m &= m - 1;                                                                              \
      if (lane < 24) wr_yuv_chain_fill(a, wbase + src, lane);                                  \
    }                                                                                          \
  }
#endif
WR_SETUP_KERNEL_YUV(wr_setup_composite_yuv)

// brush_yuv_image vertex stage (brush_yuv_image.glsl:41-93): BrushBatchKind::YuvImage — video frames drawn
// as primitives inside a picture.  The brush vertex stage, then fetch_yuv_primitive / write_uv_rect; the
// fragment and span stages are composite's (CompositeYuvShader).
WRD void wr_setup_brush_yuv_image_one(const SetupArgs& a, int idx) {
  int4 aData = *(const int4*)(a.instances + (size_t)idx * a.stride);
  QuadOut q;
  BrushVS vs;
  memset(&q, 0, sizeof q);
  wr_brush_vertex(a, aData, 1, q, vs);
  const FrameTablesDev& T = a.tabs;
  float4 data = wr_fetch(T.gpu_cache, T.n_gpu_cache, vs.ph.specific_prim_address);
  int bit_depth = (int)data.x, color_space = (int)data.y, format = (int)data.z;
  int planes = wr_yuv_planes(format);
  const TexView* tv[3] = {&a.color0, &a.color1, &a.color2};
  const int rescale = wr_yuv_rescale(format, bit_depth, tv);
  bool bad = rescale < 0 || planes == 0;
  for (int p = 0; p < planes; p++) bad = bad || !tv[p]->ptr;
  if (bad) {
    wr_yuv_reject(a, idx);
    wr_finish_setup(a, 1);
    return;
  }
  const float* lr = vs.ph.lr;
  float4 uvr[3];
  for (int p = 0; p < 3; p++) uvr[p] = p < planes ? wr_fetch(T.gpu_cache, T.n_gpu_cache, vs.ph.user_data[p]) : make_float4(0, 0, 0, 0);
  for (int kx = 0; kx < 4; kx++) {
    float fx = (vs.local_pos[kx].x - lr[0]) / (lr[2] - lr[0]);
    float fy = (vs.local_pos[kx].y - lr[1]) / (lr[3] - lr[1]);
    for (int p = 0; p < planes; p++) {
      q.interp[kx][2 * p] = ((uvr[p].z - uvr[p].x) * fx + uvr[p].x) / (float)tv[p]->w;
      q.interp[kx][2 * p + 1] = ((uvr[p].w - uvr[p].y) * fy + uvr[p].y) / (float)tv[p]->h;
    }
  }
  q.n_interp = 6;
  q.flags |= CMD_TEXTURED;
  q.col[0] = q.col[1] = q.col[2] = q.col[3] = 255;
  int unsupported = 0;
  bool ok = wr_emit_quad(a, idx, q, &unsupported);
  if (ok) {
    CmdCold* k = &a.cold[idx];
    for (int p = 0; p < 3; p++) {
      float tw = (float)tv[p]->w, th = (float)tv[p]->h;
      k->g[4 * p + 0] = (uvr[p].x + 0.5f) / tw;
      k->g[4 * p + 1] = (uvr[p].y + 0.5f) / th;
      k->g[4 * p + 2] = (uvr[p].z - 0.5f) / tw;
      k->g[4 * p + 3] = (uvr[p].w - 0.5f) / th;
    }
    wr_yuv_color_matrix(color_space, format, bit_depth, &k->g[12], &k->g[15]);
    YuvFixed m = wr_yuv_fixed_from(&k->g[12], &k->g[15], rescale);
    int* mi = (int*)(k->g + 24);
    mi[0] = m.bu; mi[1] = m.rv; mi[2] = m.gu; mi[3] = m.gv;
    mi[4] = m.y_coeff; mi[5] = m.y_bias; mi[6] = m.uv_bias; mi[7] = m.br_y_mask;
    mi[9] = (16 - rescale - 1) - 8;  // rescaleBits (swgl_ext.h:1087-1088)
    k->i[0] = format;
    k->i[1] = planes;
    k->i[2] = -1;
    k->i[3] = 0;
    k->g[32] = (a.features & WRCU_FEAT_ALPHA_PASS) ? 1.0f : 0.0f;
    wr_yuv_chain_table(a, idx, planes, tv);
  }
  wr_finish_setup(a, unsupported);
}
WR_SETUP_KERNEL_YUV(wr_setup_brush_yuv_image)

template <> struct WrRun<CompositeYuvShader> {  // brush_yuv_image draws under depth test; composite never does
  enum { n = 6 };
  WRD_MEMBER int drawn(const CompositeYuvShader::Row& r) { return r.body_len; }
};
template <> struct WrRun<CompositeYuv16Shader> : WrRun<CompositeYuvShader> {};

#ifndef WRCU_HOSTEMU
// Strip mode: with the chain table the Row holds nothing that depends on the tile (the u sums come from the
// table, v does not move along a row, the tail pixels interpolate from the span start).
template <> struct WrRowReuse<CompositeYuvShader> {
  enum { v = 1 };
  WRD_MEMBER bool ok(const CompositeYuvShader::Row& r) { return r.chain != nullptr; }
};
template <> struct WrRowReuse<CompositeYuv16Shader> : WrRowReuse<CompositeYuvShader> {};
#endif

#ifndef WRCU_HOSTEMU
// The same shader compiled for ONE resident CTA per SM (255 registers): the row state of three planes no longer
// spills (608 bytes of stack at 128 registers).  WRCU_YUV_WIDE=1 launches it; measured against the default in
// profiles/README_r02.md.
struct CompositeYuvShaderWide : CompositeYuvShader {};
template <> struct WrMinCtas<CompositeYuvShaderWide> { enum { v = 1 }; };
template <> struct WrRun<CompositeYuvShaderWide> {
  enum { n = 6 };
  WRD_MEMBER int drawn(const CompositeYuvShader::Row& r) { return r.body_len; }
};
#endif
