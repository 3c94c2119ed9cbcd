// Implicit-GEMM k x k convolution on tcgen05 for channels-last image rows (stride 1, zero padding 'same', dilation):
//
//   out[r, n] = epilogue( sum_{tap, c} g(act[pixel(r) + tap, c]) . W[n, tap * C + c] )        r over N*H*W rows
//
// Replaces usf_im2col + usf_linear (nn.Conv2d of ConvNet2D / GatedConv, reference networks.py:61-121, 405-494) without
// materialising the gathered operand matrix (k*k*C columns per row in HBM): the A operand of every 128-row tile is built
// IN SHARED MEMORY by four gather warps -- one thread per tile row reads the k*k neighbour pixels of its row from global
// memory (128 B per pixel at C = 32; the 9-fold re-reads hit L1/L2), applies the coupling mask / the ReLU in front of the
// convolution, splits each value into tf32 hi + lo and writes both planes in the K-major 128B-swizzled layout the tensor
// core reads -- while the whole weight (k*k*C x N in two tf32 planes, 74 KB at C = N = 32, k = 3) stays resident in shared
// memory for the lifetime of the persistent CTA (loaded once by TMA).  fp32-accurate 3-term tf32 split
// (A_hi.W_hi + A_lo.W_hi + A_hi.W_lo), accumulation chains closed every `chunk_slabs` K-slabs and summed in fp32 registers
// by the epilogue warps, exactly as the 3xTF32 engine of the contraction (gemm_tc2.cuh); the fused epilogue (bias, ReLU,
// output planes) is shared.
//
// Warp roles (N <= 32: 768 threads): warp 0 weight loader (TMA, once), warp 1 MMA issuer + TMEM owner, warps 4-7
// epilogue, warps 8-23 gather (4 threads per tile row).  3 A stages of 32 KB (hi + lo) + the resident weight.
#pragma once
#include "gemm_tc.cuh"

namespace usf {
namespace convtc {

using namespace tc;

// Warp layout by tile width.  N <= 32 (the hidden convolutions of the image conditioners): 4 epilogue warps (one TMEM
// lane quarter each, all 32 columns) and 16 gather warps, 4 threads per tile row; N <= 64: 8 epilogue warps (two column
// halves) and 8 gather warps, 2 threads per row -- the register file does not hold 64 fp32 partial sums per epilogue
// thread next to 16 gather warps.
constexpr int conv_epi_warps(int bn) { return bn <= 32 ? 4 : 8; }
constexpr int conv_gather_tpr(int bn) { return bn <= 32 ? 4 : 2; }           // gather threads per tile row
constexpr int conv_gather_warp0(int bn) { return FIRST_EPI_WARP + conv_epi_warps(bn); }
constexpr int conv_threads(int bn) { return (conv_gather_warp0(bn) + BLOCK_M * conv_gather_tpr(bn) / 32) * 32; }
constexpr int MAX_A_STAGES = 8;                     // the A stage count is a launch parameter (conv_tc_stages)
constexpr int A_TILE = BLOCK_M * SLAB_BYTES;        // 16 KB per plane
constexpr int A_STAGE_BYTES = 2 * A_TILE;           // hi + lo

__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int BLOCK_N>
__global__ void __launch_bounds__(conv_threads(BLOCK_N), 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_w_lo,
               const float* __restrict__ act, long long ld_act, long long M, int H, int W, int Cin, int ksize, int dil,
               const float* __restrict__ mask, int relu_in, int N, int K, int chunk_slabs, Epilogue ep, int A_STAGES) {
  using C = Config<BLOCK_N, 3, false>;
  constexpr int B_SLAB = BLOCK_N * SLAB_BYTES;      // one K-slab of one weight plane (multiple of 1024 B)
  constexpr int CONV_EPI_WARPS = conv_epi_warps(BLOCK_N), GATHER_TPR = conv_gather_tpr(BLOCK_N);
  constexpr int GATHER_WARP0 = conv_gather_warp0(BLOCK_N);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int k_slabs = (K + 31) / 32;
  const uint32_t w_base = smem_base + A_STAGES * A_STAGE_BYTES;
  const uint32_t bar_base = w_base + (uint32_t)k_slabs * 2u * B_SLAB;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (A_STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * A_STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * A_STAGES + 2 + s); };
  const uint32_t wfull_bar = bar_base + 8u * (2 * A_STAGES + 4);
  const uint32_t tmem_slot = bar_base + 8u * (2 * A_STAGES + 5);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long n_tiles = (M + BLOCK_M - 1) / BLOCK_M;
  if (chunk_slabs <= 0 || chunk_slabs > k_slabs) chunk_slabs = k_slabs;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_w);
    prefetch_tmap(&tm_w_lo);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < A_STAGES; ++s) { mbar_init(full_bar(s), BLOCK_M * GATHER_TPR / 32); mbar_init(empty_bar(s), 1); }
      for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), CONV_EPI_WARPS); }
      mbar_init(wfull_bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== weight loader: the whole [N, K] weight, both planes, once =====================
    if (lane == 0) {
      mbar_expect_tx(wfull_bar, (uint32_t)k_slabs * 2u * B_SLAB);
      for (int ks = 0; ks < k_slabs; ++ks) {
        tma_load_2d(w_base + (uint32_t)ks * 2u * B_SLAB, &tm_w, wfull_bar, ks * 32, 0);
        tma_load_2d(w_base + (uint32_t)ks * 2u * B_SLAB + B_SLAB, &tm_w_lo, wfull_bar, ks * 32, 0);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    mbar_wait(wfull_bar, 0);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      for (int ks0 = 0; ks0 < k_slabs; ks0 += chunk_slabs) {
        const int ks1 = ks0 + chunk_slabs < k_slabs ? ks0 + chunk_slabs : k_slabs;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * C::ACC_STRIDE;
        for (int ks = ks0; ks < ks1; ++ks) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          if (lane == 0) {
            const uint32_t sa = smem_base + stage * A_STAGE_BYTES;
            const uint32_t sb = w_base + (uint32_t)ks * 2u * B_SLAB;
            const uint64_t da_hi = make_smem_desc(sa), da_lo = make_smem_desc(sa + A_TILE);
            const uint64_t db_hi = make_smem_desc(sb), db_lo = make_smem_desc(sb + B_SLAB);
#pragma unroll
            for (int k = 0; k < SLAB_BYTES / UMMA_K_BYTES; ++k) {   // small terms first
              const uint64_t koff = (uint64_t)((k * UMMA_K_BYTES) >> 4);
              umma<false>(da_lo + koff, db_hi + koff, tmem_d, C::IDESC, (ks > ks0 || k > 0) ? 1u : 0u);
              umma<false>(da_hi + koff, db_lo + koff, tmem_d, C::IDESC, 1u);
            }
#pragma unroll
            for (int k = 0; k < SLAB_BYTES / UMMA_K_BYTES; ++k) {
              const uint64_t koff = (uint64_t)((k * UMMA_K_BYTES) >> 4);
              umma<false>(da_hi + koff, db_hi + koff, tmem_d, C::IDESC, 1u);
            }
            umma_commit(empty_bar(stage));
            if (ks == ks1 - 1) umma_commit(tfull_bar(acc));
          }
          __syncwarp();
          if (++stage == A_STAGES) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= GATHER_WARP0) {
    // ===================== gather warps: GATHER_TPR threads build one row of every A tile =====================
    // (i) the tap geometry is resolved ONCE per (thread, K-slab): C_in % 16 == 0 puts the thread's 16-byte chunks inside
    // one tap, i.e. one border test and one source pointer per item, advanced incrementally from slab to slab;
    // (ii) software pipeline over the flat sequence of (tile, K-slab) work items with two register sets: the global loads
    // of item i+1 are in flight while item i is converted and stored (the stores are asm volatile; loads and stores of
    // ONE item in one loop would serialise on the load latency, and so would a register copy between the sets).
    constexpr int CPT = 8 / GATHER_TPR;                       // 16-byte chunks of the 128-byte slab row per thread
    const int g = threadIdx.x - GATHER_WARP0 * 32;
    const int t = g / GATHER_TPR, q = g % GATHER_TPR;         // tile row, first chunk = q * CPT
    const int HW = H * W, half = ksize >> 1;
    const uint32_t row_off = (uint32_t)(t >> 3) * 1024u + (uint32_t)(t & 7) * 128u;
    uint32_t col[CPT];                                        // swizzled 16-byte slots of this thread's chunks
#pragma unroll
    for (int j = 0; j < CPT; ++j) col[j] = ((uint32_t)(q * CPT + j) ^ (uint32_t)(t & 7)) << 4;
    int stage = 0;
    uint32_t phase = 0;
    struct Item {                       // (tile, slab) + where this thread's chunks come from (nullptr: zeros)
      long long tile;
      int ks, ty, tx, c;                // tap (row, column) and first channel of the thread's chunks in slab ks
      const float* src;
      const float* msk;
    };
    const int k4_0 = q * (CPT * 4);     // the thread's first column in slab 0 -> its tap / channel (divisions once)
    const int tap_0 = k4_0 / Cin, c_0 = k4_0 - tap_0 * Cin, ty_0 = tap_0 / ksize, tx_0 = tap_0 - ty_0 * ksize;
    long long r = 0;                    // this thread's pixel in the tile being LOADED
    int h = 0, w = 0;
    auto pixel = [&](long long tile) {
      r = tile * BLOCK_M + t;
      const int p = r < M ? (int)(r % HW) : 0;
      h = p / W;
      w = p - h * W;
    };
    auto resolve = [&](Item& it) {      // tap of the thread's chunks in slab it.ks -> source / mask pointers
      const int dh = (it.ty - half) * dil, dw = (it.tx - half) * dil;
      const bool inside = r < M && it.ty < ksize && (unsigned)(h + dh) < (unsigned)H && (unsigned)(w + dw) < (unsigned)W;
      it.src = inside ? act + (r + dh * W + dw) * ld_act + it.c : nullptr;
      it.msk = (inside && mask) ? mask + (long long)((h + dh) * W + (w + dw)) * Cin + it.c : nullptr;
    };
    auto load_item = [&](const Item& it, float4 (&v)[CPT]) {
#pragma unroll
      for (int j = 0; j < CPT; ++j)
        v[j] = it.src ? *reinterpret_cast<const float4*>(it.src + 4 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto store_item = [&](const Item& it, const float4 (&src)[CPT]) {
      mbar_wait(empty_bar(stage), phase ^ 1);
      const uint32_t sa = smem_base + stage * A_STAGE_BYTES + row_off;
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        float4 v = src[j];
        if (it.msk) {                                        // tiny (H*W*C floats): L1 resident
          const float4 m = __ldg(reinterpret_cast<const float4*>(it.msk + 4 * j));
          v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
        }
        if (relu_in) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        const float hx = tf32_round(v.x), hy = tf32_round(v.y), hz = tf32_round(v.z), hw_ = tf32_round(v.w);
        st_shared_v4(sa + col[j], hx, hy, hz, hw_);
        st_shared_v4(sa + A_TILE + col[j], tf32_round(v.x - hx), tf32_round(v.y - hy), tf32_round(v.z - hz), tf32_round(v.w - hw_));
      }
      fence_proxy_async();                 // generic-proxy stores -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) mbar_arrive(full_bar(stage));             // one arrival per warp
      if (++stage == A_STAGES) { stage = 0; phase ^= 1; }
    };
    auto advance = [&](const Item& a, Item& b) {             // next work item of this CTA (refreshes the pixel per tile)
      if (a.ks + 1 < k_slabs) {
        b.tile = a.tile; b.ks = a.ks + 1; b.ty = a.ty; b.tx = a.tx;
        b.c = a.c + 32;                                       // 32 columns further: at most two taps on (C_in >= 16)
        while (b.c >= Cin) { b.c -= Cin; if (++b.tx == ksize) { b.tx = 0; ++b.ty; } }
      } else {
        b.tile = a.tile + gridDim.x; b.ks = 0; b.ty = ty_0; b.tx = tx_0; b.c = c_0;
        pixel(b.tile);
      }
      resolve(b);
    };
    float4 va[CPT], vb[CPT];
    Item ia, ib;
    ia.tile = blockIdx.x;
    ia.ks = 0;
    ia.ty = ty_0; ia.tx = tx_0; ia.c = c_0;
    pixel(ia.tile);
    resolve(ia);
    if (ia.tile < n_tiles) load_item(ia, va);
    while (ia.tile < n_tiles) {
      advance(ia, ib);
      if (ib.tile < n_tiles) load_item(ib, vb);
      store_item(ia, va);
      if (ib.tile >= n_tiles) break;
      advance(ib, ia);
      if (ia.tile < n_tiles) load_item(ia, va);
      store_item(ib, vb);
    }
  } else if (warp >= FIRST_EPI_WARP && warp < FIRST_EPI_WARP + CONV_EPI_WARPS) {
    // ===================== epilogue warps (as gemm_tc.cuh) =====================
    if (CONV_EPI_WARPS == 4)
      epilogue_loop<C, BLOCK_N>(0, warp & 3, lane, tmem_base, tfull_bar(0), tempty_bar(0), n_tiles, 1, k_slabs, chunk_slabs, M, N, ep);
    else if (warp < FIRST_EPI_WARP + 4)
      epilogue_loop<C, C::HALF0>(0, warp & 3, lane, tmem_base, tfull_bar(0), tempty_bar(0), n_tiles, 1, k_slabs, chunk_slabs, M, N, ep);
    else
      epilogue_loop<C, C::HALF1>(C::HALF0, warp & 3, lane, tmem_base, tfull_bar(0), tempty_bar(0), n_tiles, 1, k_slabs, chunk_slabs, M, N, ep);
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::TMEM_COLS) : "memory");
  }
}

}  // namespace convtc

struct ConvGeom {
  const float* act;
  long long ld_act;
  int H, W, Cin, ksize, dil;
  const float* mask;
  int relu_in;
};

// A stages: measured on the 32 -> 32 channel 3x3 convolution (B200): 3 stages 388 us, 4 stages 427 us
// (the per-slab hand-over, not the pipeline depth, bounds the kernel), so 3 it is.  0 = the shape does not fit.
inline int conv_tc_stages(int block_n, int K) {
  const long long w = (long long)((K + 31) / 32) * 2 * block_n * tc::SLAB_BYTES;
  return 3 * convtc::A_STAGE_BYTES + w + 1024 + 256 <= 227 * 1024 ? 3 : 0;
}
inline size_t conv_tc_smem_bytes(int block_n, int K) {
  return (size_t)conv_tc_stages(block_n, K) * convtc::A_STAGE_BYTES + (size_t)((K + 31) / 32) * 2 * block_n * tc::SLAB_BYTES + 1024 + 256;
}

// K-slabs (32 tf32 elements each) per TMEM accumulation chain of the convolution: 3 = 96 elements per chain (the chain
// hand-over is what bounds the kernel: 388 us at 2, 363 us at 3, 356 us at 9 slabs for the 3x3 32->32 convolution; the
// truncation bias of a 96-element chain is ~5e-7 relative, measured 5e-6 at 1024 elements)
constexpr int CONV_CHUNK_SLABS = 3;
template <int BLOCK_N>
int launch_conv_tc_cfg(const usf_linear_args* a, const ConvGeom& g, const Epilogue& ep, cudaStream_t st) {
  auto kern = convtc::conv_tc_kernel<BLOCK_N>;
  const size_t smem = conv_tc_smem_bytes(BLOCK_N, a->K);
  static size_t attr_bytes_dev[MAX_DEVICES] = {0};
  size_t& attr_bytes = attr_bytes_dev[current_device_slot()];
  if (smem > attr_bytes) {
    USF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_bytes = smem;
  }
  CUtensorMap mw, mwl;
  int rc;
  if ((rc = make_operand_map(&mw, a->w, a->N, a->K, a->ldw, BLOCK_N, 0))) return rc;
  if ((rc = make_operand_map(&mwl, a->w_lo, a->N, a->K, a->ldw, BLOCK_N, 0))) return rc;
  const long long tiles = (a->M + tc::BLOCK_M - 1) / tc::BLOCK_M;
  const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
  kern<<<grid, convtc::conv_threads(BLOCK_N), smem, st>>>(mw, mwl, g.act, g.ld_act, a->M, g.H, g.W, g.Cin, g.ksize, g.dil, g.mask,
                                                 g.relu_in, a->N, a->K, CONV_CHUNK_SLABS, ep, conv_tc_stages(BLOCK_N, a->K));
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int launch_conv_tc(const usf_linear_args* a, const ConvGeom& g, const Epilogue& ep, cudaStream_t st);

}  // namespace usf
