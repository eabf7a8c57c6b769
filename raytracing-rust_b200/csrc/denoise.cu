// ptb200 — on-device denoiser of the C ABI (include/ptb200.h "denoiser"): the spatial part of SVGF (Schied et al. 2017,
// §4.3-4.5) over the beauty accumulator and the AOV sums of ptb_render_aov. The header states the definition; the CPU
// restatement is oracle/denoise_api.cpp, in the same order of operations.
//
// Launches on the context's stream, all one thread per pixel, no atomics:
//   k_denoise_prepare   sums -> irradiance e = c / max(a, 1e-3) and the guide records (normal | depth, coverage, depth
//                       gradient)
//   k_denoise_variance  7x7 feature-weighted moments of ℓ(e) -> [e.rgb | var]
//   k_denoise_atrous    one launch per level (step 2^i), ping-pong [e.rgb | var]; the last level multiplies the albedo
//                       back in and stores RGB
// ptb_denoise_temporal (SVGF §4.1-4.2, CPU restatement oracle/temporal_api.cpp) runs k_denoise_prepare, then
//   k_temporal_integrate  reprojects the context's history through the motion sums and integrates colour and moments
//   k_temporal_variance   [e_int | var]: the moments' variance from 4 frames of history on, the 7x7 estimate before
// and the same levels, level 0 writing the next history (k_temporal_modulate stores RGB when it is also the last).
// A tap reads 36 bytes: [e.rgb | var] and [n.xyz | z] (16 B each) and the coverage α (4 B). The taps go through L1; a
// shared-memory tile for the small steps was not built.
#include <cmath>
#include <utility>

#include "ptb_internal.h"

namespace ptb {
namespace {

constexpr float kLog2e = 1.44269504088896341f;
constexpr uint32_t kMaxLevels = 10;
constexpr int kBlockX = 16, kBlockY = 8;

struct DenoiseSigmas {
  float l, n, z;
};

__device__ __forceinline__ float luminance(float r, float g, float b) { return (0.2126f * r + 0.7152f * g) + 0.0722f * b; }

// the à-trous taps h = (3/8, 1/4, 1/16) by |d|
__device__ __forceinline__ float h_tap(int d) { return d == 0 ? 0.375f : d == 1 || d == -1 ? 0.25f : 0.0625f; }

__device__ __forceinline__ bool zero3(const float4& v) { return v.x == 0.0f && v.y == 0.0f && v.z == 0.0f; }

// σ_n * log2(max(0, n_p·n_q)), 0 when both normals are zero (the caller drops a tap where exactly one is)
__device__ __forceinline__ float normal_term(const float4& np, const float4& nq, bool zero_p, float sigma_n) {
  if (zero_p) return 0.0f;
  const float dot = (np.x * nq.x + np.y * nq.y) + np.z * nq.z;
  return sigma_n * log2f(fmaxf(0.0f, dot));
}

// depth of pixel j (depth sum / coverage sum) and whether it counts for the gradient (coverage sum > 0)
__device__ __forceinline__ float pixel_depth(const float4* __restrict__ aov, size_t j, bool& covered) {
  const float cov = aov[2 * j].w;
  covered = cov > 0.0f;
  return covered ? aov[2 * j + 1].w / cov : 0.0f;
}

// the smaller-magnitude one-sided difference over the covered in-image neighbours (forward on a tie), 0 if neither counts
__device__ __forceinline__ float depth_gradient(float z, float z_fwd, bool fwd, float z_bwd, bool bwd) {
  const float f = z_fwd - z, b = z - z_bwd;
  if (fwd && bwd) return fabsf(f) <= fabsf(b) ? f : b;
  if (fwd) return f;
  if (bwd) return b;
  return 0.0f;
}

__global__ void k_denoise_prepare(const float* __restrict__ beauty, const float4* __restrict__ aov, int w, int h,
                                  float inv_b, float s_a, float4* __restrict__ e_out, float4* __restrict__ nz_out,
                                  float* __restrict__ alpha_out, float2* __restrict__ grad_out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const size_t i = (size_t)y * w + x;
  const float4 s0 = aov[2 * i], s1 = aov[2 * i + 1];
  const float dr = fmaxf(s0.x / s_a, 1e-3f), dg = fmaxf(s0.y / s_a, 1e-3f), db = fmaxf(s0.z / s_a, 1e-3f);
  e_out[i] = make_float4(beauty[3 * i + 0] * inv_b / dr, beauty[3 * i + 1] * inv_b / dg, beauty[3 * i + 2] * inv_b / db, 0.0f);
  const float len = sqrtf((s1.x * s1.x + s1.y * s1.y) + s1.z * s1.z);
  float4 nz = len > 0.0f ? make_float4(s1.x / len, s1.y / len, s1.z / len, 0.0f) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  bool cov_p;
  nz.w = pixel_depth(aov, i, cov_p);
  nz_out[i] = nz;
  alpha_out[i] = s0.w / s_a;
  bool cf = false, cb = false;
  float zf = 0.0f, zb = 0.0f;
  if (x + 1 < w) zf = pixel_depth(aov, i + 1, cf);
  if (x > 0) zb = pixel_depth(aov, i - 1, cb);
  const float gx = depth_gradient(nz.w, zf, cf, zb, cb);
  cf = cb = false;
  if (y + 1 < h) zf = pixel_depth(aov, i + w, cf);
  if (y > 0) zb = pixel_depth(aov, i - w, cb);
  grad_out[i] = make_float2(gx, depth_gradient(nz.w, zf, cf, zb, cb));
}

// SVGF's spatial variance estimate of pixel (x, y) over `e_in`: 7x7 feature-weighted moments of ℓ(e)
__device__ __forceinline__ float spatial_variance(const float4* __restrict__ e_in, const float4* __restrict__ nz,
                                                  const float* __restrict__ alpha, const float2* __restrict__ grad, int w,
                                                  int h, DenoiseSigmas sg, int x, int y, size_t i, const float4& ep) {
  const float4 np = nz[i];
  const float ap = alpha[i], lp = luminance(ep.x, ep.y, ep.z);
  const float2 gp = grad[i];
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
        const float4 nq = nz[j];
        if (zp != zero3(nq)) continue;
        const float4 eq = e_in[j];
        lq = luminance(eq.x, eq.y, eq.z);
        const float d_z = (sg.z * fabsf(gp.x * (float)dx + gp.y * (float)dy) + dz_base) + 1e-6f;
        const float t_z = fabsf(np.w - nq.w) / d_z;
        wq = (1.0f - fabsf(ap - alpha[j])) * exp2f(normal_term(np, nq, zp, sg.n) - t_z * kLog2e);
      }
      sw += wq;
      m1 += wq * lq;
      m2 += wq * (lq * lq);
    }
  }
  const float mu1 = m1 / sw, mu2 = m2 / sw;
  return fmaxf(0.0f, mu2 - mu1 * mu1);
}

__global__ void __launch_bounds__(kBlockX * kBlockY)
k_denoise_variance(const float4* __restrict__ e_in, const float4* __restrict__ nz, const float* __restrict__ alpha,
                   const float2* __restrict__ grad, int w, int h, DenoiseSigmas sg, float4* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const size_t i = (size_t)y * w + x;
  const float4 ep = e_in[i];
  out[i] = make_float4(ep.x, ep.y, ep.z, spatial_variance(e_in, nz, alpha, grad, w, h, sg, x, y, i, ep));
}

// one à-trous level; `rgb` != nullptr marks the last one: e * max(albedo, 1e-3) goes there instead of `out`
__global__ void __launch_bounds__(kBlockX * kBlockY)
k_denoise_atrous(const float4* __restrict__ in, const float4* __restrict__ nz, const float* __restrict__ alpha,
                 const float2* __restrict__ grad, int w, int h, int step, DenoiseSigmas sg, float4* __restrict__ out,
                 float* __restrict__ rgb, const float4* __restrict__ aov, float s_a) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const size_t i = (size_t)y * w + x;
  const float4 ep = in[i], np = nz[i];
  const float ap = alpha[i], lp = luminance(ep.x, ep.y, ep.z);
  const float2 gp = grad[i];
  const bool zp = zero3(np);
  // 3x3 Gaussian of the variance, normalised over the neighbours inside the image
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
  const float d_l = sg.l * sqrtf(gs / ks) + 1e-10f;
  const float dz_base = 1e-3f * np.w;
  float sr = 0.0f, sgr = 0.0f, sb = 0.0f, sw = 0.0f, sv = 0.0f;
  for (int dy = -2; dy <= 2; ++dy) {
    const int yy = y + dy * step;
    if (yy < 0 || yy >= h) continue;
    for (int dx = -2; dx <= 2; ++dx) {
      const int xx = x + dx * step;
      if (xx < 0 || xx >= w) continue;
      float wq;
      float4 eq;
      if (dx == 0 && dy == 0) {
        wq = 0.140625f;  // h(0)^2
        eq = ep;
      } else {
        const size_t j = (size_t)yy * w + xx;
        const float4 nq = nz[j];
        if (zp != zero3(nq)) continue;
        eq = in[j];
        const float lq = luminance(eq.x, eq.y, eq.z);
        const float d_z = (sg.z * fabsf(gp.x * (float)(dx * step) + gp.y * (float)(dy * step)) + dz_base) + 1e-6f;
        const float t = fabsf(np.w - nq.w) / d_z + fabsf(lp - lq) / d_l;
        wq = (h_tap(dx) * h_tap(dy)) * (1.0f - fabsf(ap - alpha[j])) * exp2f(normal_term(np, nq, zp, sg.n) - t * kLog2e);
      }
      sr += wq * eq.x;
      sgr += wq * eq.y;
      sb += wq * eq.z;
      sw += wq;
      sv += (wq * wq) * eq.w;
    }
  }
  const float er = sr / sw, eg = sgr / sw, eb = sb / sw;
  if (rgb) {
    const float4 s0 = aov[2 * i];
    rgb[3 * i + 0] = er * fmaxf(s0.x / s_a, 1e-3f);
    rgb[3 * i + 1] = eg * fmaxf(s0.y / s_a, 1e-3f);
    rgb[3 * i + 2] = eb * fmaxf(s0.z / s_a, 1e-3f);
  } else {
    out[i] = make_float4(er, eg, eb, sv / (sw * sw));
  }
}

// ---- temporal accumulation (SVGF §4.1-4.2, include/ptb200.h "temporal denoiser")
struct TemporalParams {
  float alpha_c, alpha_m, max_len;
  int have_history;
};
constexpr float kTapNormal = 0.9f, kTapDepthGrad = 4.0f, kTapDepthRel = 0.02f, kMinHistoryWeight = 0.01f;

// Reprojects the history through the pixel's mean motion (bilinear taps, each kept only when its guides match) and
// integrates: e_int = (1 - a_c) e_hist + a_c e, moments alike. e_int -> e_out (w = 0), [m1, m2, len, 0] -> m_out.
__global__ void __launch_bounds__(kBlockX * kBlockY)
k_temporal_integrate(const float4* __restrict__ e_in, const float4* __restrict__ motion, const float4* __restrict__ nz,
                     const float4* __restrict__ h_e, const float4* __restrict__ h_m, const float4* __restrict__ h_nz,
                     const float* __restrict__ h_alpha, const float2* __restrict__ h_grad, int w, int h, TemporalParams tp,
                     float4* __restrict__ e_out, float4* __restrict__ m_out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const size_t i = (size_t)y * w + x;
  const float4 e = e_in[i], mot = motion[i], np = nz[i];
  float er = 0.0f, eg = 0.0f, eb = 0.0f, m1 = 0.0f, m2 = 0.0f, len_h = 0.0f;
  if (tp.have_history && mot.w > 0.0f) {
    const float qx = (float)x + mot.x / mot.w, qy = (float)y + mot.y / mot.w, tq = mot.z / mot.w;
    const float x0 = floorf(qx), y0 = floorf(qy), fx = qx - x0, fy = qy - y0;
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, s1 = 0.0f, s2 = 0.0f, sl = 0.0f;
    for (int dy = 0; dy <= 1; ++dy) {
      for (int dx = 0; dx <= 1; ++dx) {
        const float wq = (dx ? fx : 1.0f - fx) * (dy ? fy : 1.0f - fy);
        const float xq = x0 + (float)dx, yq = y0 + (float)dy;
        if (!(wq > 0.0f) || !(xq >= 0.0f && xq < (float)w && yq >= 0.0f && yq < (float)h)) continue;
        const size_t j = (size_t)yq * w + (size_t)xq;
        if (!(h_alpha[j] > 0.0f)) continue;
        const float4 nq = h_nz[j];
        if (zero3(nq) || (np.x * nq.x + np.y * nq.y) + np.z * nq.z < kTapNormal) continue;
        const float2 gq = h_grad[j];
        if (fabsf(tq - nq.w) > kTapDepthGrad * (fabsf(gq.x) + fabsf(gq.y)) + kTapDepthRel * nq.w) continue;
        const float4 ce = h_e[j], cm = h_m[j];
        sw += wq;
        sr += wq * ce.x;
        sg += wq * ce.y;
        sb += wq * ce.z;
        s1 += wq * cm.x;
        s2 += wq * cm.y;
        sl += wq * cm.z;
      }
    }
    if (sw > kMinHistoryWeight) {
      er = sr / sw; eg = sg / sw; eb = sb / sw;
      m1 = s1 / sw; m2 = s2 / sw; len_h = sl / sw;
    }
  }
  const float len = fminf(len_h + 1.0f, tp.max_len);
  const float ac = fmaxf(tp.alpha_c, 1.0f / len), am = fmaxf(tp.alpha_m, 1.0f / len);
  e_out[i] = make_float4((1.0f - ac) * er + ac * e.x, (1.0f - ac) * eg + ac * e.y, (1.0f - ac) * eb + ac * e.z, 0.0f);
  const float l = luminance(e.x, e.y, e.z);
  m_out[i] = make_float4((1.0f - am) * m1 + am * l, (1.0f - am) * m2 + am * (l * l), len, 0.0f);
}

// [e_int | var]: the integrated moments' variance once 4 frames are in the history, the spatial estimate before
__global__ void __launch_bounds__(kBlockX * kBlockY)
k_temporal_variance(const float4* __restrict__ e_in, const float4* __restrict__ m, const float4* __restrict__ nz,
                    const float* __restrict__ alpha, const float2* __restrict__ grad, int w, int h, DenoiseSigmas sg,
                    float4* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const size_t i = (size_t)y * w + x;
  const float4 ep = e_in[i], mi = m[i];
  const float var = mi.z >= 4.0f ? fmaxf(0.0f, mi.y - mi.x * mi.x) : spatial_variance(e_in, nz, alpha, grad, w, h, sg, x, y, i, ep);
  out[i] = make_float4(ep.x, ep.y, ep.z, var);
}

// rgb = e * max(albedo, 1e-3): the last level's output when level 0 (kept as history) is also the last
__global__ void k_temporal_modulate(const float4* __restrict__ e, const float4* __restrict__ aov, size_t npix, float s_a,
                                    float* __restrict__ rgb) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const float4 ei = e[i], s0 = aov[2 * i];
  rgb[3 * i + 0] = ei.x * fmaxf(s0.x / s_a, 1e-3f);
  rgb[3 * i + 1] = ei.y * fmaxf(s0.y / s_a, 1e-3f);
  rgb[3 * i + 2] = ei.z * fmaxf(s0.z / s_a, 1e-3f);
}

int32_t check_denoise(Ctx* c, const ptb_denoise_opts* opts) {
  if (!opts) return set_error(c, PTB_ERR_INVALID, "null denoise opts");
  if (!c->d_accum.p) return set_error(c, PTB_ERR_INVALID, "nothing rendered yet");
  if (!c->d_aov.p) return set_error(c, PTB_ERR_INVALID, "no AOV rendered yet");
  if (c->accum_w != c->aov_w || c->accum_h != c->aov_h)
    return set_error(c, PTB_ERR_INVALID, "the beauty image is %ux%u but the AOVs are %ux%u", c->accum_w, c->accum_h,
                     c->aov_w, c->aov_h);
  if (c->accum_samples == 0) return set_error(c, PTB_ERR_INVALID, "the beauty accumulator holds no samples");
  if (c->aov_samples == 0) return set_error(c, PTB_ERR_INVALID, "the AOV accumulator holds no samples");
  if (opts->iterations > kMaxLevels)
    return set_error(c, PTB_ERR_INVALID, "iterations must be <= %u (got %u)", kMaxLevels, opts->iterations);
  const struct { const char* name; float v; } sig[3] = {
      {"sigma_luminance", opts->sigma_luminance}, {"sigma_normal", opts->sigma_normal}, {"sigma_depth", opts->sigma_depth}};
  for (const auto& s : sig)
    if (!(s.v >= 0.0f) || std::isinf(s.v)) return set_error(c, PTB_ERR_INVALID, "%s must be finite and >= 0 (got %g)", s.name, (double)s.v);
  if (opts->flags != 0) return set_error(c, PTB_ERR_INVALID, "denoise flags must be 0 (got 0x%x)", opts->flags);
  return PTB_OK;
}

// opts checked; writes W*H*3 floats to the device buffer `rgb`
// the scratch at the beauty image's size
int32_t ensure_denoise_scratch(Ctx* c) {
  const uint32_t w = c->accum_w, h = c->accum_h;
  const size_t npix = (size_t)w * h;
  if (c->dn_w != w || c->dn_h != h || !c->d_dn_nz.p) {
    PTB_CUDA_TRY(c, c->d_dn_e[0].alloc(npix * sizeof(float4)));
    PTB_CUDA_TRY(c, c->d_dn_e[1].alloc(npix * sizeof(float4)));
    PTB_CUDA_TRY(c, c->d_dn_nz.alloc(npix * sizeof(float4)));
    PTB_CUDA_TRY(c, c->d_dn_alpha.alloc(npix * sizeof(float)));
    PTB_CUDA_TRY(c, c->d_dn_grad.alloc(npix * sizeof(float2)));
    c->dn_w = w;
    c->dn_h = h;
  }
  return PTB_OK;
}

DenoiseSigmas sigmas_of(const ptb_denoise_opts& o) {
  return DenoiseSigmas{o.sigma_luminance != 0.0f ? o.sigma_luminance : 4.0f, o.sigma_normal != 0.0f ? o.sigma_normal : 128.0f,
                       o.sigma_depth != 0.0f ? o.sigma_depth : 1.0f};
}

int32_t launch_denoise(Ctx* c, const ptb_denoise_opts& o, float* rgb) {
  const uint32_t w = c->accum_w, h = c->accum_h;
  const int32_t rc = ensure_denoise_scratch(c);
  if (rc != PTB_OK) return rc;
  const uint32_t levels = o.iterations ? o.iterations : 5u;
  const DenoiseSigmas sg = sigmas_of(o);
  const float s_a = (float)c->aov_samples;
  float4* e[2] = {c->d_dn_e[0].as<float4>(), c->d_dn_e[1].as<float4>()};
  const float4* aov = c->d_aov.as<float4>();
  float4* nz = c->d_dn_nz.as<float4>();
  float* alpha = c->d_dn_alpha.as<float>();
  float2* grad = c->d_dn_grad.as<float2>();
  const dim3 block(kBlockX, kBlockY), grid((w + kBlockX - 1) / kBlockX, (h + kBlockY - 1) / kBlockY);
  k_denoise_prepare<<<grid, block, 0, c->stream>>>(c->d_accum.as<float>(), aov, (int)w, (int)h, 1.0f / (float)c->accum_samples,
                                                   s_a, e[0], nz, alpha, grad);
  k_denoise_variance<<<grid, block, 0, c->stream>>>(e[0], nz, alpha, grad, (int)w, (int)h, sg, e[1]);
  for (uint32_t l = 0; l < levels; ++l) {
    const bool last = l + 1 == levels;
    const float4* src = e[(l + 1) & 1u];
    k_denoise_atrous<<<grid, block, 0, c->stream>>>(src, nz, alpha, grad, (int)w, (int)h, 1 << l, sg, e[l & 1u],
                                                    last ? rgb : nullptr, aov, s_a);
  }
  c->stats.kernel_launches += 2 + levels;
  PTB_CUDA_TRY(c, cudaGetLastError());
  return PTB_OK;
}

int32_t check_temporal(Ctx* c, const ptb_temporal_opts* opts) {
  if (!opts) return set_error(c, PTB_ERR_INVALID, "null temporal opts");
  const int32_t rc = check_denoise(c, &opts->spatial);
  if (rc != PTB_OK) return rc;
  const struct { const char* name; float v; } al[2] = {{"alpha_color", opts->alpha_color}, {"alpha_moments", opts->alpha_moments}};
  for (const auto& a : al)
    if (!(a.v == 0.0f || (a.v > 0.0f && a.v <= 1.0f)))
      return set_error(c, PTB_ERR_INVALID, "%s must be in (0, 1] or 0 (got %g)", a.name, (double)a.v);
  if (opts->max_history > 255) return set_error(c, PTB_ERR_INVALID, "max_history must be <= 255 (got %u)", opts->max_history);
  if (opts->flags != 0) return set_error(c, PTB_ERR_INVALID, "temporal flags must be 0 (got 0x%x)", opts->flags);
  return PTB_OK;
}

void swap_buf(DevBuf& a, DevBuf& b) {
  std::swap(a.p, b.p);
  std::swap(a.bytes, b.bytes);
}

// opts checked; writes W*H*3 floats to the device buffer `rgb` and makes this frame the history
int32_t launch_temporal(Ctx* c, const ptb_temporal_opts& o, float* rgb) {
  const uint32_t w = c->accum_w, h = c->accum_h;
  const size_t npix = (size_t)w * h;
  int32_t rc = ensure_denoise_scratch(c);
  if (rc != PTB_OK) return rc;
  if (c->th_w != w || c->th_h != h || !c->d_th_nz.p) {
    c->have_history = false;
    for (DevBuf* b : {&c->d_th_e[0], &c->d_th_e[1], &c->d_th_m[0], &c->d_th_m[1], &c->d_th_nz})
      PTB_CUDA_TRY(c, b->alloc(npix * sizeof(float4)));
    PTB_CUDA_TRY(c, c->d_th_alpha.alloc(npix * sizeof(float)));
    PTB_CUDA_TRY(c, c->d_th_grad.alloc(npix * sizeof(float2)));
    c->th_w = w;
    c->th_h = h;
  }
  const uint32_t levels = o.spatial.iterations ? o.spatial.iterations : 5u;
  const DenoiseSigmas sg = sigmas_of(o.spatial);
  const TemporalParams tp{o.alpha_color != 0.0f ? o.alpha_color : 0.2f, o.alpha_moments != 0.0f ? o.alpha_moments : 0.2f,
                          (float)(o.max_history ? o.max_history : 32u), c->have_history ? 1 : 0};
  const float s_a = (float)c->aov_samples;
  const uint32_t cur = c->th_cur, nxt = cur ^ 1u;
  float4* e[2] = {c->d_dn_e[0].as<float4>(), c->d_dn_e[1].as<float4>()};
  float4* hist_out = c->d_th_e[nxt].as<float4>();
  const float4* aov = c->d_aov.as<float4>();
  float4* nz = c->d_dn_nz.as<float4>();
  float* alpha = c->d_dn_alpha.as<float>();
  float2* grad = c->d_dn_grad.as<float2>();
  const dim3 block(kBlockX, kBlockY), grid((w + kBlockX - 1) / kBlockX, (h + kBlockY - 1) / kBlockY);
  k_denoise_prepare<<<grid, block, 0, c->stream>>>(c->d_accum.as<float>(), aov, (int)w, (int)h, 1.0f / (float)c->accum_samples,
                                                   s_a, e[0], nz, alpha, grad);
  k_temporal_integrate<<<grid, block, 0, c->stream>>>(e[0], c->d_motion.as<float4>(), nz, c->d_th_e[cur].as<float4>(),
                                                      c->d_th_m[cur].as<float4>(), c->d_th_nz.as<float4>(),
                                                      c->d_th_alpha.as<float>(), c->d_th_grad.as<float2>(), (int)w, (int)h, tp,
                                                      e[1], c->d_th_m[nxt].as<float4>());
  k_temporal_variance<<<grid, block, 0, c->stream>>>(e[1], c->d_th_m[nxt].as<float4>(), nz, alpha, grad, (int)w, (int)h, sg, e[0]);
  // level 0 writes the next history; later levels ping-pong through the scratch from there
  k_denoise_atrous<<<grid, block, 0, c->stream>>>(e[0], nz, alpha, grad, (int)w, (int)h, 1, sg, hist_out, nullptr, aov, s_a);
  for (uint32_t l = 1; l < levels; ++l) {
    const bool last = l + 1 == levels;
    const float4* src = l == 1 ? hist_out : e[(l + 1) & 1u];
    k_denoise_atrous<<<grid, block, 0, c->stream>>>(src, nz, alpha, grad, (int)w, (int)h, 1 << l, sg, e[l & 1u],
                                                    last ? rgb : nullptr, aov, s_a);
  }
  if (levels == 1)
    k_temporal_modulate<<<(unsigned)((npix + 255) / 256), 256, 0, c->stream>>>(hist_out, aov, npix, s_a, rgb);
  c->stats.kernel_launches += 3 + levels + (levels == 1 ? 1 : 0);
  PTB_CUDA_TRY(c, cudaGetLastError());
  // this frame's guides become the history's; the old history's buffers are the next call's scratch
  swap_buf(c->d_dn_nz, c->d_th_nz);
  swap_buf(c->d_dn_alpha, c->d_th_alpha);
  swap_buf(c->d_dn_grad, c->d_th_grad);
  c->th_cur = nxt;
  c->have_history = true;
  return PTB_OK;
}

}  // namespace
}  // namespace ptb

using namespace ptb;

extern "C" {

int32_t ptb_denoise(ptb_ctx* ctx, const ptb_denoise_opts* opts, float* rgb, size_t n_floats) {
  if (!ctx) return PTB_ERR_INVALID;
  Ctx* c = &ctx->c;
  if (cudaSetDevice(c->device) != cudaSuccess) return set_error(c, PTB_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  int32_t rc = check_denoise(c, opts);
  if (rc != PTB_OK) return rc;
  const size_t n = (size_t)c->accum_w * c->accum_h * 3;
  if (!rgb || n_floats != n) return set_error(c, PTB_ERR_INVALID, "denoise expects %zu floats", n);
  PTB_CUDA_TRY(c, c->d_hits.reserve(n * sizeof(float)));
  rc = launch_denoise(c, *opts, c->d_hits.as<float>());
  if (rc != PTB_OK) return rc;
  PTB_CUDA_TRY(c, cudaMemcpyAsync(rgb, c->d_hits.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

int32_t ptb_denoise_device(ptb_ctx* ctx, const ptb_denoise_opts* opts, void* d_rgb) {
  if (!ctx) return PTB_ERR_INVALID;
  Ctx* c = &ctx->c;
  if (cudaSetDevice(c->device) != cudaSuccess) return set_error(c, PTB_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  const int32_t rc = check_denoise(c, opts);
  if (rc != PTB_OK) return rc;
  if (!d_rgb) return set_error(c, PTB_ERR_INVALID, "null device output");
  return launch_denoise(c, *opts, static_cast<float*>(d_rgb));
}

int32_t ptb_denoise_temporal(ptb_ctx* ctx, const ptb_temporal_opts* opts, float* rgb, size_t n_floats) {
  if (!ctx) return PTB_ERR_INVALID;
  Ctx* c = &ctx->c;
  if (cudaSetDevice(c->device) != cudaSuccess) return set_error(c, PTB_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  int32_t rc = check_temporal(c, opts);
  if (rc != PTB_OK) return rc;
  const size_t n = (size_t)c->accum_w * c->accum_h * 3;
  if (!rgb || n_floats != n) return set_error(c, PTB_ERR_INVALID, "denoise expects %zu floats", n);
  PTB_CUDA_TRY(c, c->d_hits.reserve(n * sizeof(float)));
  rc = launch_temporal(c, *opts, c->d_hits.as<float>());
  if (rc != PTB_OK) return rc;
  PTB_CUDA_TRY(c, cudaMemcpyAsync(rgb, c->d_hits.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

int32_t ptb_denoise_temporal_device(ptb_ctx* ctx, const ptb_temporal_opts* opts, void* d_rgb) {
  if (!ctx) return PTB_ERR_INVALID;
  Ctx* c = &ctx->c;
  if (cudaSetDevice(c->device) != cudaSuccess) return set_error(c, PTB_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  const int32_t rc = check_temporal(c, opts);
  if (rc != PTB_OK) return rc;
  if (!d_rgb) return set_error(c, PTB_ERR_INVALID, "null device output");
  return launch_temporal(c, *opts, static_cast<float*>(d_rgb));
}

int32_t ptb_denoise_temporal_reset(ptb_ctx* ctx) {
  if (!ctx) return PTB_ERR_INVALID;
  ctx->c.have_history = false;
  return PTB_OK;
}

}  // extern "C"
