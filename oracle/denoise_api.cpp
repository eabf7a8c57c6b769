// ORACLE — TEST INFRASTRUCTURE ONLY.
// The denoiser of ptb_denoise (include/ptb200.h "denoiser": the spatial part of SVGF, Schied et al. 2017 §4.3-4.5)
// restated on the CPU in f32, operation by operation in the device's order (raytracing-rust_b200/csrc/denoise.cu), built
// without FMA contraction. Only exp2f, log2f (glibc against the device's) may differ; sqrtf and every division are IEEE
// on both sides.
//
// Inputs are the raw sums: beauty (H, W, 3) of s_b samples; AOV (H, W, 8) = albedo.rgb, coverage, normal.xyz, depth of
// s_a samples (oracle/aov_oracle.py's layout, the device's records). Output (H, W, 3).
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <thread>
#include <vector>

namespace {

constexpr float kLog2e = 1.44269504088896341f;

struct V4 {
  float x = 0, y = 0, z = 0, w = 0;
};

float luminance(float r, float g, float b) { return (0.2126f * r + 0.7152f * g) + 0.0722f * b; }
float h_tap(int d) { return d == 0 ? 0.375f : d == 1 || d == -1 ? 0.25f : 0.0625f; }
bool zero3(const V4& v) { return v.x == 0.0f && v.y == 0.0f && v.z == 0.0f; }

float normal_term(const V4& np, const V4& nq, bool zero_p, float sigma_n) {
  if (zero_p) return 0.0f;
  const float dot = (np.x * nq.x + np.y * nq.y) + np.z * nq.z;
  return sigma_n * log2f(std::fmax(0.0f, dot));
}

struct Image {
  int w, h;
  const float* aov;  // 8 floats per pixel
  float depth(size_t j, bool& covered) const {
    const float cov = aov[8 * j + 3];
    covered = cov > 0.0f;
    return covered ? aov[8 * j + 7] / cov : 0.0f;
  }
};

float depth_gradient(float z, float z_fwd, bool fwd, float z_bwd, bool bwd) {
  const float f = z_fwd - z, b = z - z_bwd;
  if (fwd && bwd) return std::fabs(f) <= std::fabs(b) ? f : b;
  if (fwd) return f;
  if (bwd) return b;
  return 0.0f;
}

// fn(y) for every row; rows are independent within a pass, so the result does not depend on the thread count
template <class F>
void for_rows(int h, unsigned threads, const F& fn) {
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < threads; ++t)
    pool.emplace_back([&, t]() {
      for (int y = (int)t; y < h; y += (int)threads) fn(y);
    });
  for (auto& th : pool) th.join();
}

}  // namespace

extern "C" int ora_denoise(const float* beauty, const float* aov, uint32_t width, uint32_t height, uint64_t s_b, uint64_t s_a,
                           uint32_t iterations, float sigma_l, float sigma_n, float sigma_z, float* out, uint32_t threads) {
  if (width == 0 || height == 0 || s_b == 0 || s_a == 0 || iterations > 10) return 1;
  const int w = (int)width, h = (int)height;
  const size_t npix = (size_t)w * h;
  const uint32_t levels = iterations ? iterations : 5u;
  if (sigma_l == 0.0f) sigma_l = 4.0f;
  if (sigma_n == 0.0f) sigma_n = 128.0f;
  if (sigma_z == 0.0f) sigma_z = 1.0f;
  const float inv_b = 1.0f / (float)s_b, sa = (float)s_a;
  const Image im{w, h, aov};
  if (threads == 0) threads = std::max(1u, std::thread::hardware_concurrency());

  // prepare
  std::vector<V4> e0(npix), e1(npix), nz(npix);
  std::vector<float> alpha(npix), gx(npix), gy(npix);
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
      nz[i] = n;
      alpha[i] = s[3] / sa;
      bool cf = false, cb = false;
      float zf = 0.0f, zb = 0.0f;
      if (x + 1 < w) zf = im.depth(i + 1, cf);
      if (x > 0) zb = im.depth(i - 1, cb);
      gx[i] = depth_gradient(n.w, zf, cf, zb, cb);
      cf = cb = false;
      zf = zb = 0.0f;
      if (y + 1 < h) zf = im.depth(i + w, cf);
      if (y > 0) zb = im.depth(i - w, cb);
      gy[i] = depth_gradient(n.w, zf, cf, zb, cb);
    }
  });

  // variance: 7x7 moments of the luminance, weighted by w_α * w_n * w_z; the centre's weight is 1
  for_rows(h, threads, [&](int y) {
    for (int x = 0; x < w; ++x) {
      const size_t i = (size_t)y * w + x;
      const V4 ep = e0[i], np = nz[i];
      const float ap = alpha[i], lp = luminance(ep.x, ep.y, ep.z);
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
            const V4 nq = nz[j];
            if (zp != zero3(nq)) continue;
            const V4 eq = e0[j];
            lq = luminance(eq.x, eq.y, eq.z);
            const float d_z = (sigma_z * std::fabs(gx[i] * (float)dx + gy[i] * (float)dy) + dz_base) + 1e-6f;
            const float t_z = std::fabs(np.w - nq.w) / d_z;
            wq = (1.0f - std::fabs(ap - alpha[j])) * exp2f(normal_term(np, nq, zp, sigma_n) - t_z * kLog2e);
          }
          sw += wq;
          m1 += wq * lq;
          m2 += wq * (lq * lq);
        }
      }
      const float mu1 = m1 / sw, mu2 = m2 / sw;
      e1[i] = V4{ep.x, ep.y, ep.z, std::fmax(0.0f, mu2 - mu1 * mu1)};
    }
  });

  // à-trous levels, ping-pong: the variance's output feeds level 0
  std::vector<V4>* src = &e1;
  std::vector<V4>* dst = &e0;
  for (uint32_t l = 0; l < levels; ++l) {
    const int step = 1 << l;
    const bool last = l + 1 == levels;
    const std::vector<V4>& in = *src;
    std::vector<V4>& res = *dst;
    for_rows(h, threads, [&](int y) {
      for (int x = 0; x < w; ++x) {
        const size_t i = (size_t)y * w + x;
        const V4 ep = in[i], np = nz[i];
        const float ap = alpha[i], lp = luminance(ep.x, ep.y, ep.z);
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
              const V4 nq = nz[j];
              if (zp != zero3(nq)) continue;
              eq = in[j];
              const float lq = luminance(eq.x, eq.y, eq.z);
              const float d_z = (sigma_z * std::fabs(gx[i] * (float)(dx * step) + gy[i] * (float)(dy * step)) + dz_base) + 1e-6f;
              const float t = std::fabs(np.w - nq.w) / d_z + std::fabs(lp - lq) / d_l;
              wq = (h_tap(dx) * h_tap(dy)) * (1.0f - std::fabs(ap - alpha[j])) *
                   exp2f(normal_term(np, nq, zp, sigma_n) - t * kLog2e);
            }
            sr += wq * eq.x;
            sg += wq * eq.y;
            sb += wq * eq.z;
            sw += wq;
            sv += (wq * wq) * eq.w;
          }
        }
        const float er = sr / sw, eg = sg / sw, eb = sb / sw;
        if (last) {
          const float* s = aov + 8 * i;
          out[3 * i + 0] = er * std::fmax(s[0] / sa, 1e-3f);
          out[3 * i + 1] = eg * std::fmax(s[1] / sa, 1e-3f);
          out[3 * i + 2] = eb * std::fmax(s[2] / sa, 1e-3f);
        } else {
          res[i] = V4{er, eg, eb, sv / (sw * sw)};
        }
      }
    });
    std::swap(src, dst);
  }
  return 0;
}
