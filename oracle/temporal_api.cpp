// ORACLE — TEST INFRASTRUCTURE ONLY.
// The temporal denoiser of ptb_denoise_temporal (include/ptb200.h "temporal denoiser": SVGF §4.1-4.2 in front of the
// spatial filter) restated on the CPU in f32 as ONE stateless step: the sums and the history in, the image and the next
// history out. Operation by operation in the device's order (raytracing-rust_b200/csrc/denoise.cu), built without FMA
// contraction, over denoise_api.cpp's helpers; as there only exp2f, log2f may differ from the device.
//
// Layouts (row-major, top row first): beauty (H, W, 3) sums of s_b samples; AOV (H, W, 8) sums of s_a samples; motion
// (H, W, 4) sums [Δx, Δy, t', count]; history: colour (H, W, 4) [e.rgb | -], moments (H, W, 4) [m1, m2, len, 0],
// guides nz (H, W, 4) [n.xyz | z], alpha (H, W), grad (H, W, 2) [∂x z, ∂y z].
#include "denoise_api.cpp"

namespace {

struct Guides {
  std::vector<V4> nz;
  std::vector<float> alpha, gx, gy;
};

// the 7x7 spatial variance at pixel i of `e` (k_denoise_variance)
float spatial_variance(const std::vector<V4>& e, const Guides& g, int w, int h, float sigma_n, float sigma_z, int x, int y) {
  const size_t i = (size_t)y * w + x;
  const V4 ep = e[i], np = g.nz[i];
  const float ap = g.alpha[i], lp = luminance(ep.x, ep.y, ep.z);
  const bool zp = zero3(np);
  const float dz_base = 1e-3f * np.w;
  float sw = 0.0f, m1 = 0.0f, m2 = 0.0f;
  for (int dy = -3; dy <= 3; ++dy) {
    const int yy = y + dy;
    if (yy < 0 || yy >= h) continue;
    for (int dx = -3; dx <= 3; ++dx) {
      const int xx = x + dx;
      if (xx < 0 || xx >= w) continue;
      float wq, lq;
      if (dx == 0 && dy == 0) {
        wq = 1.0f;
        lq = lp;
      } else {
        const size_t j = (size_t)yy * w + xx;
        const V4 nq = g.nz[j];
        if (zp != zero3(nq)) continue;
        const V4 eq = e[j];
        lq = luminance(eq.x, eq.y, eq.z);
        const float d_z = (sigma_z * std::fabs(g.gx[i] * (float)dx + g.gy[i] * (float)dy) + dz_base) + 1e-6f;
        const float t_z = std::fabs(np.w - nq.w) / d_z;
        wq = (1.0f - std::fabs(ap - g.alpha[j])) * exp2f(normal_term(np, nq, zp, sigma_n) - t_z * kLog2e);
      }
      sw += wq;
      m1 += wq * lq;
      m2 += wq * (lq * lq);
    }
  }
  const float mu1 = m1 / sw, mu2 = m2 / sw;
  return std::fmax(0.0f, mu2 - mu1 * mu1);
}

// one à-trous level at pixel (x, y) of `in` (k_denoise_atrous): [e' | var']
V4 atrous(const std::vector<V4>& in, const Guides& g, int w, int h, int step, float sigma_l, float sigma_n, float sigma_z,
          int x, int y) {
  const size_t i = (size_t)y * w + x;
  const V4 ep = in[i], np = g.nz[i];
  const float ap = g.alpha[i], lp = luminance(ep.x, ep.y, ep.z);
  const bool zp = zero3(np);
  float gs = 0.0f, ks = 0.0f;
  for (int dy = -1; dy <= 1; ++dy) {
    const int yy = y + dy;
    if (yy < 0 || yy >= h) continue;
    for (int dx = -1; dx <= 1; ++dx) {
      const int xx = x + dx;
      if (xx < 0 || xx >= w) continue;
      const float k = dx == 0 && dy == 0 ? 0.25f : dx == 0 || dy == 0 ? 0.125f : 0.0625f;
      gs += k * in[(size_t)yy * w + xx].w;
      ks += k;
    }
  }
  const float d_l = sigma_l * std::sqrt(gs / ks) + 1e-10f;
  const float dz_base = 1e-3f * np.w;
  float sr = 0.0f, sg = 0.0f, sb = 0.0f, sw = 0.0f, sv = 0.0f;
  for (int dy = -2; dy <= 2; ++dy) {
    const int yy = y + dy * step;
    if (yy < 0 || yy >= h) continue;
    for (int dx = -2; dx <= 2; ++dx) {
      const int xx = x + dx * step;
      if (xx < 0 || xx >= w) continue;
      float wq;
      V4 eq;
      if (dx == 0 && dy == 0) {
        wq = 0.140625f;
        eq = ep;
      } else {
        const size_t j = (size_t)yy * w + xx;
        const V4 nq = g.nz[j];
        if (zp != zero3(nq)) continue;
        eq = in[j];
        const float lq = luminance(eq.x, eq.y, eq.z);
        const float d_z = (sigma_z * std::fabs(g.gx[i] * (float)(dx * step) + g.gy[i] * (float)(dy * step)) + dz_base) + 1e-6f;
        const float t = std::fabs(np.w - nq.w) / d_z + std::fabs(lp - lq) / d_l;
        wq = (h_tap(dx) * h_tap(dy)) * (1.0f - std::fabs(ap - g.alpha[j])) * exp2f(normal_term(np, nq, zp, sigma_n) - t * kLog2e);
      }
      sr += wq * eq.x;
      sg += wq * eq.y;
      sb += wq * eq.z;
      sw += wq;
      sv += (wq * wq) * eq.w;
    }
  }
  return V4{sr / sw, sg / sw, sb / sw, sv / (sw * sw)};
}

}  // namespace

extern "C" int ora_denoise_temporal(const float* beauty, const float* aov, const float* motion, uint32_t width, uint32_t height,
                                    uint64_t s_b, uint64_t s_a, uint32_t iterations, float sigma_l, float sigma_n, float sigma_z,
                                    float alpha_c, float alpha_m, uint32_t max_history, int have_history, const float* h_e,
                                    const float* h_m, const float* h_nz, const float* h_alpha, const float* h_grad, float* out,
                                    float* o_e, float* o_m, float* o_nz, float* o_alpha, float* o_grad, uint32_t threads) {
  if (width == 0 || height == 0 || s_b == 0 || s_a == 0 || iterations > 10 || max_history > 255) return 1;
  const int w = (int)width, h = (int)height;
  const size_t npix = (size_t)w * h;
  const uint32_t levels = iterations ? iterations : 5u;
  if (sigma_l == 0.0f) sigma_l = 4.0f;
  if (sigma_n == 0.0f) sigma_n = 128.0f;
  if (sigma_z == 0.0f) sigma_z = 1.0f;
  if (alpha_c == 0.0f) alpha_c = 0.2f;
  if (alpha_m == 0.0f) alpha_m = 0.2f;
  const float max_len = (float)(max_history ? max_history : 32u);
  const float inv_b = 1.0f / (float)s_b, sa = (float)s_a;
  const Image im{w, h, aov};
  if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());

  // prepare (k_denoise_prepare)
  std::vector<V4> e0(npix), e1(npix), hist(npix), mom(npix);
  Guides g;
  g.nz.resize(npix);
  g.alpha.resize(npix);
  g.gx.resize(npix);
  g.gy.resize(npix);
  for_rows(h, threads, [&](int y) {
    for (int x = 0; x < w; ++x) {
      const size_t i = (size_t)y * w + x;
      const float* s = aov + 8 * i;
      const float dr = std::fmax(s[0] / sa, 1e-3f), dg = std::fmax(s[1] / sa, 1e-3f), db = std::fmax(s[2] / sa, 1e-3f);
      e0[i] = V4{beauty[3 * i + 0] * inv_b / dr, beauty[3 * i + 1] * inv_b / dg, beauty[3 * i + 2] * inv_b / db, 0.0f};
      const float len = std::sqrt((s[4] * s[4] + s[5] * s[5]) + s[6] * s[6]);
      V4 n;
      if (len > 0.0f) n = V4{s[4] / len, s[5] / len, s[6] / len, 0.0f};
      bool cov_p;
      n.w = im.depth(i, cov_p);
      g.nz[i] = n;
      g.alpha[i] = s[3] / sa;
      bool cf = false, cb = false;
      float zf = 0.0f, zb = 0.0f;
      if (x + 1 < w) zf = im.depth(i + 1, cf);
      if (x > 0) zb = im.depth(i - 1, cb);
      g.gx[i] = depth_gradient(n.w, zf, cf, zb, cb);
      cf = cb = false;
      zf = zb = 0.0f;
      if (y + 1 < h) zf = im.depth(i + w, cf);
      if (y > 0) zb = im.depth(i - w, cb);
      g.gy[i] = depth_gradient(n.w, zf, cf, zb, cb);
    }
  });

  // reproject + integrate (k_temporal_integrate) -> e1 = [e_int | 0], mom = [m1, m2, len, 0]
  for_rows(h, threads, [&](int y) {
    for (int x = 0; x < w; ++x) {
      const size_t i = (size_t)y * w + x;
      const V4 e = e0[i], np = g.nz[i];
      const float* mot = motion + 4 * i;
      float er = 0.0f, eg = 0.0f, eb = 0.0f, m1 = 0.0f, m2 = 0.0f, len_h = 0.0f;
      if (have_history && mot[3] > 0.0f) {
        const float qx = (float)x + mot[0] / mot[3], qy = (float)y + mot[1] / mot[3], tq = mot[2] / mot[3];
        const float x0 = std::floor(qx), y0 = std::floor(qy), fx = qx - x0, fy = qy - y0;
        float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, s1 = 0.0f, s2 = 0.0f, sl = 0.0f;
        for (int dy = 0; dy <= 1; ++dy) {
          for (int dx = 0; dx <= 1; ++dx) {
            const float wq = (dx ? fx : 1.0f - fx) * (dy ? fy : 1.0f - fy);
            const float xq = x0 + (float)dx, yq = y0 + (float)dy;
            if (!(wq > 0.0f) || !(xq >= 0.0f && xq < (float)w && yq >= 0.0f && yq < (float)h)) continue;
            const size_t j = (size_t)yq * w + (size_t)xq;
            if (!(h_alpha[j] > 0.0f)) continue;
            const float* nq = h_nz + 4 * j;
            if ((nq[0] == 0.0f && nq[1] == 0.0f && nq[2] == 0.0f) || (np.x * nq[0] + np.y * nq[1]) + np.z * nq[2] < 0.9f) continue;
            const float* gq = h_grad + 2 * j;
            if (std::fabs(tq - nq[3]) > 4.0f * (std::fabs(gq[0]) + std::fabs(gq[1])) + 0.02f * nq[3]) continue;
            const float *ce = h_e + 4 * j, *cm = h_m + 4 * j;
            sw += wq;
            sr += wq * ce[0];
            sg += wq * ce[1];
            sb += wq * ce[2];
            s1 += wq * cm[0];
            s2 += wq * cm[1];
            sl += wq * cm[2];
          }
        }
        if (sw > 0.01f) {
          er = sr / sw; eg = sg / sw; eb = sb / sw;
          m1 = s1 / sw; m2 = s2 / sw; len_h = sl / sw;
        }
      }
      const float len = std::fmin(len_h + 1.0f, max_len);
      const float ac = std::fmax(alpha_c, 1.0f / len), am = std::fmax(alpha_m, 1.0f / len);
      e1[i] = V4{(1.0f - ac) * er + ac * e.x, (1.0f - ac) * eg + ac * e.y, (1.0f - ac) * eb + ac * e.z, 0.0f};
      const float l = luminance(e.x, e.y, e.z);
      mom[i] = V4{(1.0f - am) * m1 + am * l, (1.0f - am) * m2 + am * (l * l), len, 0.0f};
    }
  });

  // variance (k_temporal_variance) -> e0 = [e_int | var]
  for_rows(h, threads, [&](int y) {
    for (int x = 0; x < w; ++x) {
      const size_t i = (size_t)y * w + x;
      const V4 ep = e1[i], mi = mom[i];
      const float var = mi.z >= 4.0f ? std::fmax(0.0f, mi.y - mi.x * mi.x) : spatial_variance(e1, g, w, h, sigma_n, sigma_z, x, y);
      e0[i] = V4{ep.x, ep.y, ep.z, var};
    }
  });

  // level 0 -> the next history's colour; later levels ping-pong; the last one (or level 0 alone) is modulated out
  const std::vector<V4>* src = &e0;
  for (uint32_t l = 0; l < levels; ++l) {
    std::vector<V4>& dst = l == 0 ? hist : (l & 1u ? e1 : e0);
    const std::vector<V4>& in = *src;
    for_rows(h, threads, [&](int y) {
      for (int x = 0; x < w; ++x) dst[(size_t)y * w + x] = atrous(in, g, w, h, 1 << l, sigma_l, sigma_n, sigma_z, x, y);
    });
    src = &dst;
  }
  for (size_t i = 0; i < npix; ++i) {
    const V4 e = (*src)[i];
    const float* s = aov + 8 * i;
    out[3 * i + 0] = e.x * std::fmax(s[0] / sa, 1e-3f);
    out[3 * i + 1] = e.y * std::fmax(s[1] / sa, 1e-3f);
    out[3 * i + 2] = e.z * std::fmax(s[2] / sa, 1e-3f);
    const V4 hc = hist[i], mi = mom[i], n = g.nz[i];
    o_e[4 * i + 0] = hc.x; o_e[4 * i + 1] = hc.y; o_e[4 * i + 2] = hc.z; o_e[4 * i + 3] = hc.w;
    o_m[4 * i + 0] = mi.x; o_m[4 * i + 1] = mi.y; o_m[4 * i + 2] = mi.z; o_m[4 * i + 3] = mi.w;
    o_nz[4 * i + 0] = n.x; o_nz[4 * i + 1] = n.y; o_nz[4 * i + 2] = n.z; o_nz[4 * i + 3] = n.w;
    o_alpha[i] = g.alpha[i];
    o_grad[2 * i + 0] = g.gx[i];
    o_grad[2 * i + 1] = g.gy[i];
  }
  return 0;
}
