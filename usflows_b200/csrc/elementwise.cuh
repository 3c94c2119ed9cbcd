// HBM-bound elementwise / row-reduction kernels over [rows, d] activations.
// One warp per row-slice with 128-bit accesses when alignment allows; grid-stride over rows.
#pragma once
#include "common.cuh"

namespace usf {

struct OutPlanes {
  float* f32;
  float* hi;
  float* lo;
  __nv_bfloat16* bf16;
  long long ld_f32, ld_split, ld_bf16;
  __half* h16 = nullptr;      // fp16 split planes (x = h16 + l16 * 2^-11)
  __half* l16 = nullptr;
  long long ld_16 = 0;
  int* overflow_flag = nullptr;
};

__device__ __forceinline__ void store_planes1(const OutPlanes& o, long long r, int j, float v) {
  if (o.f32) o.f32[r * o.ld_f32 + j] = v;
  if (o.hi) {
    float h = tf32_round(v);
    o.hi[r * o.ld_split + j] = h;
    o.lo[r * o.ld_split + j] = tf32_round(v - h);
  }
  if (o.bf16) o.bf16[r * o.ld_bf16 + j] = __float2bfloat16_rn(v);
  if (o.h16) {
    __half h, l;
    f16_split(v, h, l);
    o.h16[r * o.ld_16 + j] = h;
    o.l16[r * o.ld_16 + j] = l;
    if (!(fabsf(v) <= F16_GUARD) && o.overflow_flag) *o.overflow_flag = 1;
  }
}

__device__ __forceinline__ void store_planes4(const OutPlanes& o, long long r, int j, const float (&v)[4]) {
  if (o.f32) *reinterpret_cast<float4*>(o.f32 + r * o.ld_f32 + j) = make_float4(v[0], v[1], v[2], v[3]);
  if (o.hi) {
    float h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { h[i] = tf32_round(v[i]); l[i] = tf32_round(v[i] - h[i]); }
    *reinterpret_cast<float4*>(o.hi + r * o.ld_split + j) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4*>(o.lo + r * o.ld_split + j) = make_float4(l[0], l[1], l[2], l[3]);
  }
  if (o.bf16) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&p0);
    u.y = *reinterpret_cast<uint32_t*>(&p1);
    *reinterpret_cast<uint2*>(o.bf16 + r * o.ld_bf16 + j) = u;
  }
  if (o.h16) {
    __align__(8) __half h[4];
    __align__(8) __half l[4];
    bool bad = false;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      f16_split(v[i], h[i], l[i]);
      bad = bad || !(fabsf(v[i]) <= F16_GUARD);
    }
    *reinterpret_cast<uint2*>(o.h16 + r * o.ld_16 + j) = *reinterpret_cast<const uint2*>(h);
    *reinterpret_cast<uint2*>(o.l16 + r * o.ld_16 + j) = *reinterpret_cast<const uint2*>(l);
    if (bad && o.overflow_flag) *o.overflow_flag = 1;
  }
}

// 8 consecutive values: 16-byte stores into the 16-bit planes (two 16-byte stores per 32-bit plane)
__device__ __forceinline__ void store_planes8(const OutPlanes& o, long long r, int j, const float (&v)[8]) {
  const float a[4] = {v[0], v[1], v[2], v[3]}, b[4] = {v[4], v[5], v[6], v[7]};
  if (o.f32 || o.hi) {
    OutPlanes w = o;
    w.bf16 = nullptr;
    w.h16 = nullptr;
    store_planes4(w, r, j, a);
    store_planes4(w, r, j + 4, b);
  }
  if (o.bf16) {
    __align__(16) __nv_bfloat16 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = __float2bfloat16_rn(v[i]);
    *reinterpret_cast<uint4*>(o.bf16 + r * o.ld_bf16 + j) = *reinterpret_cast<const uint4*>(t);
  }
  if (o.h16) {
    __align__(16) __half h[8];
    __align__(16) __half l[8];
    bool bad = false;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      f16_split(v[i], h[i], l[i]);
      bad = bad || !(fabsf(v[i]) <= F16_GUARD);
    }
    *reinterpret_cast<uint4*>(o.h16 + r * o.ld_16 + j) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(o.l16 + r * o.ld_16 + j) = *reinterpret_cast<const uint4*>(l);
    if (bad && o.overflow_flag) *o.overflow_flag = 1;
  }
}

inline bool planes_vec_ok(const OutPlanes& o) {
  bool ok = true;
  if (o.h16) ok = ok && aligned16(o.h16) && aligned16(o.l16) && o.ld_16 % 8 == 0;
  if (o.f32) ok = ok && aligned16(o.f32) && o.ld_f32 % 4 == 0;
  if (o.hi) ok = ok && aligned16(o.hi) && aligned16(o.lo) && o.ld_split % 4 == 0;
  if (o.bf16) ok = ok && aligned16(o.bf16) && o.ld_bf16 % 8 == 0;
  return ok;
}

// ---- Philox4x32-10 (base sampling, dequantisation noise) ------------------------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__device__ __forceinline__ void philox4x32_10(uint64_t seed, uint64_t ctr_lo, uint64_t ctr_hi, uint32_t (&out)[4]) {
  uint32_t c[4] = {(uint32_t)ctr_lo, (uint32_t)(ctr_lo >> 32), (uint32_t)ctr_hi, (uint32_t)(ctr_hi >> 32)};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}
// ---- 8-bit dequantisation (usf_dequant) -----------------------------------------------------------------
// Value k in 0..255 at flat event index j of GLOBAL row r becomes x = (k + u) / 256 with u = (2m + 1) / 2^16,
// m = Philox4x32-10(key = seed, counter = (r, j >> 2))[j & 3] >> 17 (15 bits), or u = 1/2 for the midpoint mode.
// k * 2^16 + (2m + 1) < 2^24, so x is exact in fp32 and lies strictly inside (k/256, (k+1)/256); the noise depends on
// (seed, r, j) only, so chunking, graph replay and sharding cannot change a bit.
__device__ __forceinline__ float dequant_value(uint32_t k, uint32_t rnd, int mode) {
  const uint32_t low = mode == USF_DEQUANT_MIDPOINT ? 0x8000u : (((rnd >> 17) << 1) | 1u);
  return (float)((k << 16) | low) * (1.0f / 16777216.0f);
}
// out[i] with a run-time i in 0..3, kept in registers (an indexed load would put the array in local memory)
__device__ __forceinline__ uint32_t pick4(const uint32_t (&out)[4], int i) {
  return i == 0 ? out[0] : i == 1 ? out[1] : i == 2 ? out[2] : out[3];
}

// input loaders of ingest_kernel: fp32 rows, or 8-bit rows dequantised on the fly
struct LoadF32 {
  const float* x;
  long long ldx;
  __device__ __forceinline__ void init() {}
  __device__ __forceinline__ void load4(long long r, int j, float (&v)[4]) const {
    const float4 t = __ldcs(reinterpret_cast<const float4*>(x + r * ldx + j));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  __device__ __forceinline__ float load1(long long r, int j) const { return __ldg(x + r * ldx + j); }
};
struct LoadU8 {
  const uint8_t* x;
  long long ldx;
  unsigned long long seed;
  long long row0;                  // global row of local row 0
  const long long* params;         // optional device {seed, row base}: replaces seed, adds to row0
  int mode;
  __device__ __forceinline__ void init() {
    if (params) { seed = (unsigned long long)__ldg(params); row0 += __ldg(params + 1); }
  }
  // j % 4 == 0: one 4-byte load and one Philox call for 4 elements
  __device__ __forceinline__ void load4(long long r, int j, float (&v)[4]) const {
    const uint32_t k = __ldcs(reinterpret_cast<const unsigned int*>(x + r * ldx + j));
    uint32_t rnd[4] = {0u, 0u, 0u, 0u};
    if (mode != USF_DEQUANT_MIDPOINT) philox4x32_10(seed, (uint64_t)(row0 + r), (uint64_t)(j >> 2), rnd);
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = dequant_value((k >> (8 * i)) & 0xFFu, rnd[i], mode);
  }
  __device__ __forceinline__ float load1(long long r, int j) const {
    uint32_t rnd[4] = {0u, 0u, 0u, 0u};
    if (mode != USF_DEQUANT_MIDPOINT) philox4x32_10(seed, (uint64_t)(row0 + r), (uint64_t)(j >> 2), rnd);
    return dequant_value(x[r * ldx + j], pick4(rnd, j & 3), mode);
  }
};

// ---- ingest: out = ((x / div) * mul) - sub --------------------------------------------------------
template <bool VEC, class Load>
__global__ void __launch_bounds__(256)
ingest_kernel(Load in, long long rows, int d, const float* __restrict__ dv,
              const float* __restrict__ mul, const float* __restrict__ sub, OutPlanes o) {
  griddep_launch_dependents();
  griddep_wait();
  in.init();
  if (VEC) {
    const int d4 = d >> 2;
    const long long total = rows * d4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / d4;
      const int j = (int)(i - r * d4) * 4;
      float v[4];
      in.load4(r, j, v);
      if (dv) { float4 s = __ldg(reinterpret_cast<const float4*>(dv + j)); v[0] = v[0] / s.x; v[1] = v[1] / s.y; v[2] = v[2] / s.z; v[3] = v[3] / s.w; }
      if (mul) { float4 s = __ldg(reinterpret_cast<const float4*>(mul + j)); v[0] *= s.x; v[1] *= s.y; v[2] *= s.z; v[3] *= s.w; }
      if (sub) { float4 s = __ldg(reinterpret_cast<const float4*>(sub + j)); v[0] -= s.x; v[1] -= s.y; v[2] -= s.z; v[3] -= s.w; }
      store_planes4(o, r, j, v);
    }
  } else {
    const long long total = rows * d;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / d;
      const int j = (int)(i - r * d);
      float v = in.load1(r, j);
      if (dv) v = v / __ldg(dv + j);
      if (mul) v *= __ldg(mul + j);
      if (sub) v -= __ldg(sub + j);
      store_planes1(o, r, j, v);
    }
  }
}

// ---- base log-density + row reduction ---------------------------------------------------------------
// Laplace: -log(2 s) - |z - mu| / s ; Normal: -(z-mu)^2 / (2 s^2) - log s - log sqrt(2 pi)
__device__ __forceinline__ float base_logpdf(float z, float mu, float s, int kind) {
  if (kind == USF_BASE_LAPLACE) return -logf(2.f * s) - fabsf(z - mu) / s;
  const float t = z - mu;
  return -(t * t) / (2.f * (s * s)) - logf(s) - 0.91893853320467274178f;
}

constexpr int BLP_THREADS = 256;
template <bool VEC>
__global__ void __launch_bounds__(BLP_THREADS)
base_logprob_kernel(const float* __restrict__ z, const float* __restrict__ z_lo, long long ldz, long long rows, int d,
                    const float* __restrict__ loc, const float* __restrict__ scale, int kind, float add_const,
                    float* __restrict__ out) {
  griddep_launch_dependents();
  griddep_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wpb = BLP_THREADS / 32;
  for (long long r = (long long)blockIdx.x * wpb + warp; r < rows; r += (long long)gridDim.x * wpb) {
    const float* zr = z + r * ldz;
    const float* zl = z_lo ? z_lo + r * ldz : nullptr;
    float acc = 0.f;
    if (VEC) {
      for (int j = lane * 4; j < d; j += 128) {
        float4 t = __ldcs(reinterpret_cast<const float4*>(zr + j));
        if (zl) { float4 u = __ldcs(reinterpret_cast<const float4*>(zl + j)); t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
        float4 m = __ldg(reinterpret_cast<const float4*>(loc + j));
        float4 s = __ldg(reinterpret_cast<const float4*>(scale + j));
        acc += base_logpdf(t.x, m.x, s.x, kind) + base_logpdf(t.y, m.y, s.y, kind);
        acc += base_logpdf(t.z, m.z, s.z, kind) + base_logpdf(t.w, m.w, s.w, kind);
      }
    } else {
      for (int j = lane; j < d; j += 32) {
        float t = zr[j];
        if (zl) t += zl[j];
        acc += base_logpdf(t, __ldg(loc + j), __ldg(scale + j), kind);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[r] = acc + add_const;
  }
}

// ---- base sampling --------------------------------------------------------------------------------------
// 23 random bits + 1/2: every value is exactly representable in fp32, so the result stays inside (0,1)
// (24 bits + 1/2 would round up to 1.0 for the top value and give log1p(-1) = -inf in the Laplace inverse CDF)
__device__ __forceinline__ float u01_open(uint32_t x) { return ((float)(x >> 9) + 0.5f) * (1.0f / 8388608.0f); }

// Philox key and counter base of one sampling call (usf_draw): local row r draws as GLOBAL row row0 + r, so a chunk of
// rows [r0, r1) of a larger call reproduces exactly those rows.  `params` (device {seed, row base}) replaces the seed and
// adds to row0 at run time, so one captured graph serves every chunk.
struct DrawCtr {
  unsigned long long seed, offset;
  long long row0;
  const long long* params;
  __device__ __forceinline__ void init() {
    if (params) { seed = (unsigned long long)__ldg(params); row0 += __ldg(params + 1); }
  }
};

__global__ void __launch_bounds__(256)
base_sample_kernel(long long rows, int d, const float* __restrict__ loc, const float* __restrict__ scale, int kind,
                   DrawCtr dc, OutPlanes o, int vec) {
  dc.init();
  const uint64_t seed = dc.seed, offset = dc.offset;
  const int d4 = (d + 3) >> 2;
  const long long total = rows * d4;
  const uint64_t ctr0 = (uint64_t)dc.row0 * (uint64_t)d4;        // counter of the call's row r, group g: (row0 + r) * d4 + g
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / d4;
    const int j = (int)(i - r * d4) * 4;
    uint32_t rnd[4], rnd2[4];
    philox4x32_10(seed, ctr0 + (uint64_t)i, offset, rnd);
    float e[4];
    if (kind == USF_BASE_LAPLACE) {
      // inverse CDF on u in (-1, 1): eps = -sign(u) * log1p(-|u|)  (torch.distributions.Laplace.rsample)
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float u = 2.f * u01_open(rnd[t]) - 1.f;
        e[t] = -copysignf(1.f, u) * log1pf(-fabsf(u));
      }
    } else {
      philox4x32_10(seed, ctr0 + (uint64_t)i, offset ^ 0x8000000000000000ull, rnd2);
#pragma unroll
      for (int t = 0; t < 4; t += 2) {  // Box-Muller
        const float u1 = u01_open(rnd[t]), u2 = u01_open(rnd2[t]);
        const float rad = sqrtf(-2.f * logf(u1));
        float sn, cs;
        sincospif(2.f * u2, &sn, &cs);
        e[t] = rad * cs;
        e[t + 1] = rad * sn;
      }
    }
    float v[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) v[t] = (j + t < d) ? fmaf(__ldg(scale + j + t), e[t], __ldg(loc + j + t)) : 0.f;
    if (vec && j + 3 < d) store_planes4(o, r, j, v);
    else
      for (int t = 0; t < 4 && j + t < d; ++t) store_planes1(o, r, j + t, v[t]);
  }
}

// ---- 8-bit output (usf_quantize_u8): q = min(255, max(0, floor(256 y))), NaN -> 0 ------------------------------------
// 256 y is exact in fp32, so q is the k that usf_ingest_u8 dequantises into (k/256, (k+1)/256), in either mode.
__device__ __forceinline__ uint32_t quantize_value(float y) {
  const float t = floorf(256.f * y);
  return t >= 255.f ? 255u : t >= 0.f ? (uint32_t)t : 0u;      // a NaN fails both comparisons
}

template <bool VEC>
__global__ void __launch_bounds__(256)
quantize_u8_kernel(const float* __restrict__ y, long long ldy, long long rows, int d, uint8_t* __restrict__ out, long long ldo) {
  if (VEC) {
    const int d4 = d >> 2;
    const long long total = rows * d4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / d4;
      const int j = (int)(i - r * d4) * 4;
      const float4 v = __ldcs(reinterpret_cast<const float4*>(y + r * ldy + j));
      const uint32_t q = quantize_value(v.x) | (quantize_value(v.y) << 8) | (quantize_value(v.z) << 16) | (quantize_value(v.w) << 24);
      *reinterpret_cast<uint32_t*>(out + r * ldo + j) = q;
    }
  } else {
    const long long total = rows * d;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / d;
      const int j = (int)(i - r * d);
      out[r * ldo + j] = (uint8_t)quantize_value(y[r * ldy + j]);
    }
  }
}

// ---- leaky relu / permute ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
leaky_relu_kernel(const float* __restrict__ x, long long ldx, long long rows, int d, float slope,
                  float* __restrict__ y, long long ldy, float* __restrict__ neg_count) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < rows; r += (long long)gridDim.x * 8) {
    float cnt = 0.f;
    for (int j = lane; j < d; j += 32) {
      const float v = x[r * ldx + j];
      y[r * ldy + j] = v >= 0.f ? v : v * slope;   // F.leaky_relu
      cnt += v < 0.f ? 1.f : 0.f;
    }
    if (neg_count) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      if (lane == 0) neg_count[r] = cnt;
    }
  }
}

// ---- affine coupling update (extension: the reference's coupling is additive only) ------------------------------------
// st [rows, 2h] holds the conditioner outputs of the updated features: log-scale s in columns [0, h), shift t in [h, 2h).
//   direction +1 (latent -> data): x <- x * exp(s) + t        direction -1 (data -> latent): x <- (x - t) * exp(-s)
// with s clamped to [s_min, s_max]; the row's forward log|det J| = sum_j s_j is ADDED to row_ladj[r] (one warp per row,
// shuffle reduction: the order of the sum is fixed).  x lives in whatever planes the engine mode uses and is updated in
// place.
struct XPlanes {
  float* f32;
  float* hi;
  float* lo;
  __nv_bfloat16* bf16;
  __half* h16;
  __half* l16;
  long long ld_f32, ld_split, ld_bf16, ld_16;
  int* overflow_flag;
};
__device__ __forceinline__ float xplanes_load(const XPlanes& p, long long r, int j) {
  if (p.f32) return p.f32[r * p.ld_f32 + j];
  if (p.h16) return f16_join(p.h16[r * p.ld_16 + j], p.l16[r * p.ld_16 + j]);
  if (p.hi) return p.hi[r * p.ld_split + j] + p.lo[r * p.ld_split + j];
  return __bfloat162float(p.bf16[r * p.ld_bf16 + j]);
}
__device__ __forceinline__ void xplanes_store(const XPlanes& p, long long r, int j, float v) {
  if (p.f32) p.f32[r * p.ld_f32 + j] = v;
  if (p.h16) {
    __half h, l;
    f16_split(v, h, l);
    p.h16[r * p.ld_16 + j] = h;
    p.l16[r * p.ld_16 + j] = l;
    if (!(fabsf(v) <= F16_GUARD) && p.overflow_flag) *p.overflow_flag = 1;
  }
  if (p.hi) {
    const float h = tf32_round(v);
    p.hi[r * p.ld_split + j] = h;
    p.lo[r * p.ld_split + j] = tf32_round(v - h);
  }
  if (p.bf16) p.bf16[r * p.ld_bf16 + j] = __float2bfloat16_rn(v);
}

__global__ void __launch_bounds__(256)
affine_couple_kernel(const float* __restrict__ st, long long ld_st, long long rows, int h, XPlanes x, float direction,
                     float s_min, float s_max, float* __restrict__ row_ladj) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * 8 + warp; r < rows; r += (long long)gridDim.x * 8) {
    float acc = 0.f;
    for (int j = lane; j < h; j += 32) {
      const float s = fminf(fmaxf(st[r * ld_st + j], s_min), s_max);
      const float t = st[r * ld_st + h + j];
      const float v = xplanes_load(x, r, j);
      xplanes_store(x, r, j, direction > 0.f ? fmaf(v, expf(s), t) : (v - t) * expf(-s));
      acc += s;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0 && row_ladj) row_ladj[r] += acc;
  }
}

// out[r] -= v[r]  (per-row log-determinants of affine couplings leave the density)
__global__ void __launch_bounds__(256) sub_rows_kernel(float* __restrict__ out, const float* __restrict__ v, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) out[i] -= v[i];
}

__global__ void __launch_bounds__(256)
permute_kernel(const float* __restrict__ x, long long ldx, long long rows, int d, const int* __restrict__ perm,
               float* __restrict__ y, long long ldy) {
  const long long total = rows * d;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / d;
    const int j = (int)(i - r * d);
    y[r * ldy + j] = x[r * ldx + __ldg(perm + j)];
  }
}

inline int ew_grid(long long work_items, int threads, int per_sm = 8) {
  long long blocks = (work_items + threads - 1) / threads;
  long long cap = (long long)num_sms() * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace usf
