// Image-shaped flows (in_dims = [C, H, W]; reference transforms.py:904-910 1x1-convolution mode of BlockAffineTransform,
// networks.py:405-510 ConvNet2D conditioners, flows.py:494-536 masks over [C, H, W]).
//
// Data layout: inside the layer stack an image batch [N, C, H, W] lives CHANNELS-LAST as a row matrix [N*H*W, C]:
//   * the 1x1 convolution of BlockAffineTransform is then the same row-times-matrix contraction as the flat case
//     (usf_linear over N*H*W rows), LayerNormChannels is a row LayerNorm (usf_gate_norm), and a k x k convolution is a
//     gather of the k*k neighbour rows (im2col_kernel, zero padding = 'same') followed by usf_linear with K = k*k*C_in;
//   * the base density sums over the whole event, so it reads the same memory as [N, H*W*C] with loc / scale permuted.
// Only the two ends of a pass convert between the user's NCHW tensors and this layout (layout_kernel, fused with the
// per-element ScaleTransform, transforms.py:105-125).
#pragma once
#include "elementwise.cuh"

namespace usf {

// out[n, b, a] = f(in[n, a, b]) for in [N, A, B];  f multiplies / divides by s indexed in the order of the NCHW side:
// s_on_input != 0: s[a * B + b] (the input is NCHW: A = C, B = HW), else s[b * A + a] (the output is NCHW: B = C, A = HW).
// 32 x 32 shared-memory tiles, both global accesses coalesced; 1-D grid-stride loop over (n, tile_a, tile_b).
// A uint8 input (NCHW side) is dequantised as it is read: element a * B + b of image n is event index j of global row
// dq.row0 + n (dequant_value, one Philox call per element: neighbours in a tile row may belong to different counters).
struct LayoutU8 {
  unsigned long long seed;
  long long row0;
  const long long* params;
  int mode;
};
template <class T, class OutT = float>
__global__ void __launch_bounds__(256)
layout_kernel(const T* __restrict__ in, long long N, int A, int B, const float* __restrict__ s, int s_mode, int s_on_input,
              OutT* __restrict__ out, LayoutU8 dq) {
  __shared__ float tile[32][33];
  if (sizeof(T) == 1 && dq.params) { dq.seed = (unsigned long long)__ldg(dq.params); dq.row0 += __ldg(dq.params + 1); }
  const int ta = (A + 31) >> 5, tb = (B + 31) >> 5;
  const long long tiles = N * ta * tb;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
  for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long n = t / (ta * tb);
    const int rem = (int)(t - n * (ta * tb));
    const int a0 = (rem / tb) << 5, b0 = (rem % tb) << 5;
    const T* src = in + n * (long long)A * B;
    OutT* dst = out + n * (long long)A * B;
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
      const int a = a0 + ty + i, b = b0 + tx;
      float v = 0.f;
      if (a < A && b < B) {
        const long long j = (long long)a * B + b;
        if (sizeof(T) == 1) {
          uint32_t rnd[4] = {0u, 0u, 0u, 0u};
          if (dq.mode != USF_DEQUANT_MIDPOINT) philox4x32_10(dq.seed, (uint64_t)(dq.row0 + n), (uint64_t)(j >> 2), rnd);
          v = dequant_value((uint32_t)src[j], pick4(rnd, (int)(j & 3)), dq.mode);
        } else {
          v = (float)src[j];
        }
        if (s_mode) {
          const float f = __ldg(s + (s_on_input ? (long long)a * B + b : (long long)b * A + a));
          v = s_mode == 1 ? v * f : v / f;
        }
      }
      tile[ty + i][tx] = v;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
      const int b = b0 + ty + i, a = a0 + tx;
      if (a < A && b < B) {
        if (sizeof(OutT) == 1) dst[(long long)b * A + a] = (OutT)quantize_value(tile[tx][ty + i]);
        else dst[(long long)b * A + a] = tile[tx][ty + i];
      }
    }
    __syncthreads();
  }
}

// im2col for a k x k convolution, stride 1, zero padding 'same', dilation dil, over channels-last rows:
//   out[r, (kh * k + kw) * C + c] = g(in[n, h + (kh - k/2) dil, w + (kw - k/2) dil, c])      (0 outside the image)
//   g(v) = relu ? max(v, 0) : v, after v *= mask[(h' * W + w') * C + c] when mask != NULL (coupling mask, channels-last)
// written in the operand planes of the consuming contraction.  VEC: channels per thread (1, or 4 / 8 with aligned planes
// and C % VEC == 0; 8 channels give 16-byte stores into the 16-bit operand planes).
template <int VEC>
__global__ void __launch_bounds__(256)
im2col_kernel(const float* __restrict__ in, long long ld_in, long long rows, int H, int W, int C, int k, int dil,
              const float* __restrict__ mask, int relu, OutPlanes o) {
  const int HW = H * W, kk = k * k, half = k >> 1;
  const int cg = C / VEC;
  const long long total = rows * kk * cg;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (kk * cg);
    const int rem = (int)(i - r * (kk * cg));
    const int tap = rem / cg, c = (rem - tap * cg) * VEC;
    const int p = (int)(r % HW), h = p / W, w = p - h * W;
    const int hh = h + (tap / k - half) * dil, ww = w + (tap % k - half) * dil;
    const bool inside = hh >= 0 && hh < H && ww >= 0 && ww < W;
    const long long rs = r + (long long)(hh - h) * W + (ww - w);
    const int col = tap * C + c;
    if (VEC == 8) {
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (inside) {
        const float4 t0 = *reinterpret_cast<const float4*>(in + rs * ld_in + c);
        const float4 t1 = *reinterpret_cast<const float4*>(in + rs * ld_in + c + 4);
        v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
        if (mask) {
          const float4 m0 = __ldg(reinterpret_cast<const float4*>(mask + (long long)(hh * W + ww) * C + c));
          const float4 m1 = __ldg(reinterpret_cast<const float4*>(mask + (long long)(hh * W + ww) * C + c + 4));
          v[0] *= m0.x; v[1] *= m0.y; v[2] *= m0.z; v[3] *= m0.w; v[4] *= m1.x; v[5] *= m1.y; v[6] *= m1.z; v[7] *= m1.w;
        }
        if (relu) {
#pragma unroll
          for (int q = 0; q < 8; ++q) v[q] = fmaxf(v[q], 0.f);
        }
      }
      store_planes8(o, r, col, v);
    } else if (VEC == 4) {
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (inside) {
        const float4 t = *reinterpret_cast<const float4*>(in + rs * ld_in + c);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        if (mask) {
          const float4 m = __ldg(reinterpret_cast<const float4*>(mask + (long long)(hh * W + ww) * C + c));
          v[0] *= m.x; v[1] *= m.y; v[2] *= m.z; v[3] *= m.w;
        }
        if (relu) {
#pragma unroll
          for (int q = 0; q < 4; ++q) v[q] = fmaxf(v[q], 0.f);
        }
      }
      store_planes4(o, r, col, v);
    } else {
      float v = 0.f;
      if (inside) {
        v = in[rs * ld_in + c];
        if (mask) v *= __ldg(mask + (long long)(hh * W + ww) * C + c);
        if (relu) v = fmaxf(v, 0.f);
      }
      store_planes1(o, r, col, v);
    }
  }
}

// x[r, c] += sign * g[(r mod HW) * C + c] * t[r, c]   (coupling update with a per-pixel mask, transforms.py:284-290,
// 301-306: g = 1 - mask in channels-last order)
__global__ void __launch_bounds__(256)
masked_add_kernel(float* __restrict__ x, long long ldx, const float* __restrict__ t, long long ldt, long long rows, int C,
                  int HW, const float* __restrict__ g, float sign) {
  const long long total = rows * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i - r * C);
    x[r * ldx + c] += sign * __ldg(g + (long long)(r % HW) * C + c) * t[r * ldt + c];
  }
}

}  // namespace usf
