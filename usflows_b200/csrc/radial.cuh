// Lp-radial base distribution (reference distributions.py:327-372 constructor, :501-512 log_prob, :478-499 sample,
// :514-549 log_delta_volume; norm distributions LogNormal :181-197 and GammaMM :674-707).
//
//   log p(z) = log f_R(r) - [C_p(d) + (d - 1) log r],   r = ||z - loc||_p  over the event,  p in {1, 2, inf}
//
// One warp per row: the Lp norm is a shuffle reduction over the row (HBM-bound: 4d bytes read, 4 written per row), the
// one-dimensional density of the radius is evaluated by the same warp (Gamma mixture: one component per lane).
#pragma once
#include "elementwise.cuh"

namespace usf {

constexpr int RAD_THREADS = 256;
constexpr int RAD_MAX_COMP = 128;      // Gamma mixture components (the reference's configs use 20)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Per-component constants of the radius mixture, computed once per block into shared memory.
//   USF_NORM_GAMMA_MIXTURE      params = [logits | concentration | rate]                      (K each, constrained values)
//       c_k = log w_k + a_k log b_k - lgamma(a_k)   (log w = log_softmax(logits)),  coef_k = a_k - 1
//       log f(r) = LSE_k [c_k + coef_k log r - b_k r]
//   USF_NORM_GENGAMMA_MIXTURE   params = [logits | concentration | rate | scale | power]      R = s_k S^(1 / q_k), S ~ Gamma(a_k, b_k)
//       with u = r / s_k:  log f(r) = LSE_k [c_k + log q_k - log s_k + (a_k q_k - 1) log u - b_k u^q_k]
//       (Chi: a = df / 2, b = 1 / 2, q = 2;  Weibull(lambda, k): a = b = 1, s = lambda, q = k;  HalfNormal(s): a = b = 1 / 2, q = 2)
//   USF_NORM_LOGNORMAL_MIXTURE  params = [logits | mu | sigma]
//       log f(r) = LSE_k [log w_k - log sigma_k - log sqrt(2 pi) - (log r - mu_k)^2 / (2 sigma_k^2)] - log r
struct GammaMixSmem {
  float c[RAD_MAX_COMP], am1[RAD_MAX_COMP], b[RAD_MAX_COMP], cdf[RAD_MAX_COMP];
  float a[RAD_MAX_COMP], ls[RAD_MAX_COMP], q[RAD_MAX_COMP];      // concentration (mu for log-normals), log scale, power
};
__device__ __forceinline__ void gamma_mix_prepare(GammaMixSmem& s, const float* __restrict__ params, int K, int kind) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    float m = -INFINITY;
    for (int k = lane; k < K; k += 32) m = fmaxf(m, params[k]);
    m = warp_max(m);
    float e = 0.f;
    for (int k = lane; k < K; k += 32) e += expf(params[k] - m);
    const float lse = m + logf(warp_sum(e));
    for (int k = lane; k < K; k += 32) {
      const float a = params[K + k], b = params[2 * K + k];
      s.a[k] = a;
      s.b[k] = b;
      if (kind == USF_NORM_LOGNORMAL_MIXTURE) {       // a = mu, b = sigma
        s.c[k] = params[k] - lse - logf(b) - 0.91893853320467274178f;
        s.am1[k] = 0.f; s.ls[k] = 0.f; s.q[k] = 1.f;
        continue;
      }
      s.c[k] = params[k] - lse + a * logf(b) - lgammaf(a);
      s.am1[k] = a - 1.f;
      s.ls[k] = 0.f;
      s.q[k] = 1.f;
      if (kind == USF_NORM_GENGAMMA_MIXTURE) {
        const float sc = params[3 * K + k], q = params[4 * K + k];
        s.ls[k] = logf(sc);
        s.q[k] = q;
        s.c[k] += logf(q) - s.ls[k];
        s.am1[k] = a * q - 1.f;
      }
    }
    if (lane == 0) {                       // cumulative mixture weights for sampling (K is small)
      float acc = 0.f;
      for (int k = 0; k < K; ++k) { acc += expf(params[k] - lse); s.cdf[k] = acc; }
    }
  }
  __syncthreads();
}

// log f_R(radius) evaluated by a whole warp (every lane returns the value)
__device__ __forceinline__ float radial_norm_logpdf(float radius, float logr, int norm_kind, const float* __restrict__ params,
                                                    int K, const GammaMixSmem& s, int lane) {
  if (norm_kind == USF_NORM_LOGNORMAL) {   // Normal(mu, sigma).log_prob(log r) - log r
    const float mu = __ldg(params), sg = __ldg(params + 1);
    const float u = logr - mu;
    return -(u * u) / (2.f * (sg * sg)) - logf(sg) - 0.91893853320467274178f - logr;
  }
  // term of component k; the plain Gamma mixture keeps its own expression (xlogy(a - 1, r) - b r on the radius itself)
  auto term = [&](int k) -> float {
    if (norm_kind == USF_NORM_GAMMA_MIXTURE)
      return s.c[k] + (s.am1[k] == 0.f ? 0.f : s.am1[k] * logr) - s.b[k] * radius;
    if (norm_kind == USF_NORM_LOGNORMAL_MIXTURE) {
      const float u = logr - s.a[k];
      return s.c[k] - (u * u) / (2.f * (s.b[k] * s.b[k]));
    }
    const float lu = logr - s.ls[k];
    return s.c[k] + (s.am1[k] == 0.f ? 0.f : s.am1[k] * lu) - s.b[k] * expf(s.q[k] * lu);
  };
  float m = -INFINITY;
  for (int k = lane; k < K; k += 32) m = fmaxf(m, term(k));
  m = warp_max(m);
  float e = 0.f;
  for (int k = lane; k < K; k += 32) e += expf(term(k) - m);
  const float lp = m + logf(warp_sum(e));
  return norm_kind == USF_NORM_LOGNORMAL_MIXTURE ? lp - logr : lp;
}

template <bool VEC>
__global__ void __launch_bounds__(RAD_THREADS)
radial_logprob_kernel(const float* __restrict__ z, const float* __restrict__ z_lo, long long ldz, long long rows, int d,
                      const float* __restrict__ loc, int p_kind, int norm_kind, const float* __restrict__ params, int n_comp,
                      float dv_const, float add_const, float* __restrict__ out) {
  __shared__ GammaMixSmem sm;
  if (norm_kind != USF_NORM_LOGNORMAL) gamma_mix_prepare(sm, params, n_comp, norm_kind);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wpb = RAD_THREADS / 32;
  for (long long r = (long long)blockIdx.x * wpb + warp; r < rows; r += (long long)gridDim.x * wpb) {
    const float* zr = z + r * ldz;
    const float* zl = z_lo ? z_lo + r * ldz : nullptr;
    float acc = 0.f;
    auto take = [&](float t) {
      if (p_kind == USF_LP_2) acc = fmaf(t, t, acc);
      else if (p_kind == USF_LP_1) acc += fabsf(t);
      else acc = fmaxf(acc, fabsf(t));
    };
    if (VEC) {
      for (int j = lane * 4; j < d; j += 128) {
        float4 t = __ldcs(reinterpret_cast<const float4*>(zr + j));
        if (zl) { float4 u = __ldcs(reinterpret_cast<const float4*>(zl + j)); t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
        const float4 m = __ldg(reinterpret_cast<const float4*>(loc + j));
        take(t.x - m.x); take(t.y - m.y); take(t.z - m.z); take(t.w - m.w);
      }
    } else {
      for (int j = lane; j < d; j += 32) {
        float t = zr[j];
        if (zl) t += zl[j];
        take(t - __ldg(loc + j));
      }
    }
    acc = p_kind == USF_LP_INF ? warp_max(acc) : warp_sum(acc);
    const float radius = p_kind == USF_LP_2 ? sqrtf(acc) : acc;
    const float logr = logf(radius);
    const float lp = radial_norm_logpdf(radius, logr, norm_kind, params, n_comp, sm, lane);
    if (lane == 0) out[r] = lp - (dv_const + (float)(d - 1) * logr) + add_const;
  }
}

// ---- sampling: z = loc + R * u,  R ~ norm distribution,  u uniform on the unit Lp sphere (distributions.py:270-318) ----
// Counter-based (Philox4x32-10): row r, 4-column group g uses counter (r * d4 + g, offset); the radius uses the
// counters (r, offset ^ tag).  Every value is regenerated in the second pass instead of being kept (d is unbounded).
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t ctr, uint64_t off) {
  uint32_t rnd[4];
  philox4x32_10(seed, ctr, off, rnd);
  float sn, cs;
  sincospif(2.f * u01_open(rnd[1]), &sn, &cs);
  return sqrtf(-2.f * logf(u01_open(rnd[0]))) * cs;
}

// Marsaglia-Tsang Gamma(a, 1), a >= 1; at most 64 rejection rounds (acceptance > 95% per round)
__device__ float gamma_mt(float a, uint64_t seed, uint64_t ctr, uint64_t off) {
  const float dd = a - (1.f / 3.f), c = rsqrtf(9.f * dd);
  float last = dd;
  for (uint32_t it = 0; it < 64; ++it) {
    uint32_t rnd[4];
    philox4x32_10(seed, ctr, off + 2 + it, rnd);
    float sn, cs;
    sincospif(2.f * u01_open(rnd[1]), &sn, &cs);
    const float x = sqrtf(-2.f * logf(u01_open(rnd[0]))) * cs;
    const float v0 = 1.f + c * x;
    if (v0 <= 0.f) continue;
    const float v = v0 * v0 * v0;
    last = dd * v;
    if (logf(u01_open(rnd[2])) < 0.5f * x * x + dd - dd * v + dd * logf(v)) return dd * v;
  }
  return last;
}

__global__ void __launch_bounds__(RAD_THREADS)
radial_sample_kernel(long long rows, int d, const float* __restrict__ loc, int p_kind, int norm_kind,
                     const float* __restrict__ params, int n_comp, DrawCtr dc, float* __restrict__ out, long long ldo) {
  __shared__ GammaMixSmem sm;
  if (norm_kind != USF_NORM_LOGNORMAL) gamma_mix_prepare(sm, params, n_comp, norm_kind);
  dc.init();
  const uint64_t seed = dc.seed, offset = dc.offset;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wpb = RAD_THREADS / 32;
  const int d4 = (d + 3) >> 2;
  const uint64_t RTAG = 0x4000000000000000ull;
  for (long long lr = (long long)blockIdx.x * wpb + warp; lr < rows; lr += (long long)gridDim.x * wpb) {
    const long long r = dc.row0 + lr;          // every counter below is keyed by the GLOBAL row (usf_draw)
    float* __restrict__ orow = out + lr * ldo;
    float radius = 0.f;
    int extremal = -1;
    if (lane == 0) {
      if (norm_kind == USF_NORM_LOGNORMAL) {
        radius = expf(fmaf(__ldg(params + 1), philox_normal(seed, (uint64_t)r, offset ^ RTAG), __ldg(params)));
      } else {
        uint32_t rnd[4];
        philox4x32_10(seed, (uint64_t)r, offset ^ RTAG, rnd);
        const float u = u01_open(rnd[0]);
        int k = 0;
        while (k + 1 < n_comp && u > sm.cdf[k]) ++k;
        const float a = sm.a[k], b = sm.b[k];
        if (norm_kind == USF_NORM_LOGNORMAL_MIXTURE) {          // a = mu_k, b = sigma_k
          radius = expf(fmaf(b, philox_normal(seed, (uint64_t)r, (offset ^ RTAG) + 1), a));
        } else {
          float g;
          if (a >= 1.f) g = gamma_mt(a, seed, (uint64_t)r, (offset ^ RTAG) + 1);
          else g = gamma_mt(a + 1.f, seed, (uint64_t)r, (offset ^ RTAG) + 1) * powf(u01_open(rnd[1]), 1.f / a);   // boost
          radius = g / b;
          if (norm_kind == USF_NORM_GENGAMMA_MIXTURE)           // R = s_k S^(1 / q_k)
            radius = expf(sm.ls[k]) * (sm.q[k] == 2.f ? sqrtf(radius) : powf(radius, 1.f / sm.q[k]));
        }
      }
      if (p_kind == USF_LP_INF) {
        uint32_t rnd[4];
        philox4x32_10(seed, (uint64_t)r, (offset ^ RTAG) + 0x100, rnd);
        extremal = min(d - 1, (int)(u01_open(rnd[0]) * (float)d));
      }
    }
    radius = __shfl_sync(0xffffffffu, radius, 0);
    extremal = __shfl_sync(0xffffffffu, extremal, 0);
    auto draw = [&](int g, float (&e)[4]) {
      uint32_t rnd[4];
      philox4x32_10(seed, (uint64_t)r * d4 + g, offset, rnd);
      if (p_kind == USF_LP_2) {              // standard normals (two Box-Muller pairs), normalised below
#pragma unroll
        for (int t = 0; t < 4; t += 2) {
          const float rad = sqrtf(-2.f * logf(u01_open(rnd[t])));
          float sn, cs;
          sincospif(2.f * u01_open(rnd[t + 1]), &sn, &cs);
          e[t] = rad * cs;
          e[t + 1] = rad * sn;
        }
      } else if (p_kind == USF_LP_1) {       // Dirichlet(1,..,1) = normalised exponentials, random signs
#pragma unroll
        for (int t = 0; t < 4; ++t) e[t] = ((rnd[t] & 1u) ? -1.f : 1.f) * -logf(u01_open(rnd[t]));
      } else {                                // uniform on [-1, 1], one coordinate pinned to +1 (as the reference)
#pragma unroll
        for (int t = 0; t < 4; ++t) e[t] = 2.f * u01_open(rnd[t]) - 1.f;
      }
    };
    float nrm = 1.f;
    if (p_kind != USF_LP_INF) {
      float acc = 0.f;
      for (int g = lane; g < d4; g += 32) {
        float e[4];
        draw(g, e);
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (g * 4 + t < d) acc += p_kind == USF_LP_2 ? e[t] * e[t] : fabsf(e[t]);
      }
      acc = warp_sum(acc);
      nrm = p_kind == USF_LP_2 ? sqrtf(acc) : acc;
    }
    const float mul = radius / nrm;
    for (int g = lane; g < d4; g += 32) {
      float e[4];
      draw(g, e);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int j = g * 4 + t;
        if (j < d) orow[j] = fmaf(mul, j == extremal ? 1.f : e[t], __ldg(loc + j));
      }
    }
  }
}

}  // namespace usf
