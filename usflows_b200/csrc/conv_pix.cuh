// k x k convolution of the image conditioners (networks.ConvNet2D / GatedConv, reference networks.py:61-121, 405-494) over
// channels-last PIXEL PLANES, with no gather threads at all: the operand tile of every tap is ONE 4-D TMA box.
//
// Data format ("pixel planes"): an activation with <= 32 channels is stored as [N*H*W, 64] fp16 -- per pixel 32 high
// halves | 32 low halves' (x = hi + lo' 2^-11, the fp16 split of the flat engine, missing channels zero) = 128 B, exactly
// one K-major 128B-swizzled operand row.  The tensor map sees it as [N, H, W, 64]; the box (64, W, HR, IMGS) at
// coordinates (0, dx, h0 + dy, n0) is the operand tile of tap (dy, dx) for IMGS whole images (or HR image rows of one
// image) -- rows in (n, h, w) order, zero padding 'same' and the batch / image tails by the hardware's out-of-bounds fill.
// A CTA tile is 256 rows (two M = 128 MMA tiles: 5 of the 7 x 7 MNIST images = 245 rows); the weight (per tap [32 out,
// 32 hi | 32 lo' in] = 4 KB) is resident for the life of the persistent CTA.  Per tap and MMA tile six kind::f16 MMAs
// (K = 16): the two cross terms pair the lo' half of one operand row with the hi half of the other (independent
// descriptors into the same 128-byte rows), then hi.hi; a chain of `chain_taps` taps issues its cross terms first and
// folds them in with scale-input-d 2^-11 at the first hi.hi product, as gemm_tc2.cuh; chains are summed in fp32
// registers by the epilogue warps.
//
// Two epilogues; two threads (of two warps) per pixel, 16 channels each -- the LayerNormChannels partial sums of a pixel
// meet in shared memory -- moving their rows through a per-pair staging block so that global accesses are coalesced:
//   plain : v = conv + b  [ReLU] [LayerNorm]  -> fp32 rows and / or pixel planes ([ReLU] on the planes), or the masked
//           coupling update x[r, c] += sign * (1 - mask)[pixel, c] * v[c] of transforms.py:284-290 (last convolution)
//   gated : u = relu(conv + b) is re-encoded into a shared-memory operand tile and contracted IN THE SAME KERNEL with the
//           1 x 1 convolution [val | gate] = W2 u + b2 (N = 64, second TMEM accumulator), then
//           y <- LayerNorm(relu(y + val * sigmoid(gate))) on the fp32 residual stream in place, and its pixel planes
//           -- GatedConv + ReLU + LayerNormChannels of a ConvNet2D block: one launch instead of three.
#pragma once
#include "gemm_tc.cuh"

namespace usf {

struct PixArgs {
  long long rows;                       // n_images * H * W
  long long n_tiles;
  int n_images, H, W, HW;
  int ksize, dil, taps;
  int imgs, hr, tiles_per_img;          // tile geometry: imgs whole images (tiles_per_img == 1) or hr image rows
  int chain_taps, stages, gate_at;
  unsigned box_bytes;
  int gated;
  const float* bias1;                   // [32]
  int n1, relu1;
  const float* gamma;                   // LayerNorm over the n1 channels (nullptr: none)
  const float* beta;
  float eps;
  float* out_f32;                       // plain: fp32 rows out (optional); gated: the residual stream (in / out)
  long long ld_f32;
  __half* out16;                        // pixel planes of the result (optional)
  int relu_planes;
  float* x;                             // plain: coupling update in place (optional)
  long long ldx;
  const float* inv_mask;
  float sign;
  int c_x;
  const float* bias2;                   // gated: [64]
  int post_relu;
  int* overflow_flag;
};

namespace convpix {

using namespace tc;

constexpr int MT = 2;                               // M = 128 MMA tiles per CTA tile
constexpr int TILE_ROWS = MT * BLOCK_M;
constexpr int PIX_BYTES = 128;
constexpr int A_STAGE = TILE_ROWS * PIX_BYTES;      // 32 KB
constexpr int A_MT = BLOCK_M * PIX_BYTES;           // 16 KB: second MMA tile of a stage
constexpr int W1_TAP = 32 * PIX_BYTES;              // 4 KB per tap
constexpr int W2_BYTES = 64 * PIX_BYTES;            // 8 KB
constexpr int MAX_STAGES = 6;
constexpr int PIX_EPI_WARPS = 16;                   // two warps per 32-row block: each thread owns 16 channels of one pixel
constexpr int PIX_THREADS = (FIRST_EPI_WARP + PIX_EPI_WARPS) * 32;
constexpr int NBUF = 4;                             // TMEM accumulators of the k x k convolution (chains in flight: the MMA
                                                    // issuer runs a whole tile ahead of the epilogue warps)
constexpr int ACC2_COL = NBUF * 64;                 // gate accumulator: 2 MMA tiles x 64 columns
constexpr int TMEM_COLS = 512;                      // [0,256): NBUF x 2 MMA tiles x 32; [256,384): gate
constexpr uint32_t IDESC_N32 = (1u << 4) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);   // f16 x f16 -> f32
constexpr uint32_t IDESC_N64 = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
constexpr uint64_t KOFF_LO = 64 >> 4;               // the lo' half of an operand row starts 64 B in
constexpr uint64_t KOFF_K1 = 32 >> 4;               // second K = 16 step of a half

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void umma_f16(uint64_t da, uint64_t db, uint32_t tmem_d, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D = A.B + D * 2^-11
__device__ __forceinline__ void umma_f16_scale11(uint64_t da, uint64_t db, uint32_t tmem_d, uint32_t idesc) {
  const uint32_t z = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p, 11;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(1u), "r"(z)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void st_shared_u4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// 8 consecutive channels -> 8 high halves + 8 low halves' (16 B each); returns whether a value left the fp16 range
__device__ __forceinline__ bool split8(const float* v, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
  float big = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half2 hh = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    const float2 f = __half22float2(hh);
    const __half2 ll = __floats2half2_rn((v[2 * i] - f.x) * F16_LO_SCALE, (v[2 * i + 1] - f.y) * F16_LO_SCALE);
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = *reinterpret_cast<const uint32_t*>(&ll);
    big = fmaxf(big, fmaxf(fabsf(v[2 * i]), fabsf(v[2 * i + 1])));
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
  return !(big <= F16_GUARD);
}

struct Tile {
  int n0, h0, nvalid;
  long long row0;
};
__device__ __forceinline__ Tile decode_tile(const PixArgs& p, long long tile) {
  Tile t;
  if (p.tiles_per_img == 1) {
    t.n0 = (int)(tile * p.imgs);
    t.h0 = 0;
    const int left = p.n_images - t.n0;
    t.nvalid = (left < p.imgs ? left : p.imgs) * p.HW;
    t.row0 = (long long)t.n0 * p.HW;
  } else {
    t.n0 = (int)(tile / p.tiles_per_img);
    t.h0 = (int)(tile % p.tiles_per_img) * p.hr;
    const int left = p.H - t.h0;
    t.nvalid = (left < p.hr ? left : p.hr) * p.W;
    t.row0 = (long long)t.n0 * p.HW + (long long)t.h0 * p.W;
  }
  return t;
}

// ---- staging block of a warp pair (32 rows x 128 B of shared memory, 16-byte chunks XOR-swizzled by row & 7 -- the operand
// layout of the tensor core, so the same block is the warp's part of the gate's operand tile): the epilogue thread of
// row `lane` writes / reads its 128 bytes there, and the warp moves the block to / from global memory with 512
// contiguous bytes per instruction (a thread storing its own row directly touches 32 different 128-byte lines per
// instruction: 5 700 cycles per tile for the two outputs, measured on a B200).
__device__ __forceinline__ uint4 ld_shared_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void stage_write_chunk(uint32_t stage, int lane, int c, uint4 v) {
  st_shared_u4(stage + (uint32_t)lane * 128u + ((uint32_t)(c ^ (lane & 7)) << 4), v);
}
__device__ __forceinline__ uint4 stage_read_chunk(uint32_t stage, int lane, int c) {
  return ld_shared_u4(stage + (uint32_t)lane * 128u + ((uint32_t)(c ^ (lane & 7)) << 4));
}
// ---- half rows: the two warps of a pair share one staging block; the thread of (row, half) owns channels 16*half .. +15
__device__ __forceinline__ void pair_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
// 16 fp32 channels = chunks 4*half .. 4*half + 3 of the row
__device__ __forceinline__ void stage_write_f32_half(uint32_t stage, int lane, int half, const float (&v)[16]) {
#pragma unroll
  for (int c = 0; c < 4; ++c)
    stage_write_chunk(stage, lane, 4 * half + c, make_uint4(__float_as_uint(v[4 * c]), __float_as_uint(v[4 * c + 1]),
                                                            __float_as_uint(v[4 * c + 2]), __float_as_uint(v[4 * c + 3])));
}
__device__ __forceinline__ void stage_read_f32_half(uint32_t stage, int lane, int half, float (&v)[16]) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint4 u = stage_read_chunk(stage, lane, 4 * half + c);
    v[4 * c] = __uint_as_float(u.x); v[4 * c + 1] = __uint_as_float(u.y);
    v[4 * c + 2] = __uint_as_float(u.z); v[4 * c + 3] = __uint_as_float(u.w);
  }
}
// 16 channels as pixel planes: high halves = chunks 2*half, 2*half + 1; low halves' = chunks 4 + 2*half, 5 + 2*half
template <bool RELU>
__device__ __forceinline__ bool stage_write_planes_half(uint32_t stage, int lane, int half, const float (&v)[16]) {
  bool bad = false;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    float t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t[i] = RELU ? fmaxf(v[8 * c + i], 0.f) : v[8 * c + i];
    uint4 hi, lo;
    bad |= split8(t, hi, lo);
    stage_write_chunk(stage, lane, 2 * half + c, hi);
    stage_write_chunk(stage, lane, 4 + 2 * half + c, lo);
  }
  return bad;
}
// rows 16*half .. 16*half + 15 of the block -> global rows at `pitch` bytes, `nch` 16-byte chunks per row, rows < nrows
// only (the other 16 rows are the partner warp's); lane l moves chunk l % 8 of row 4i + l / 8: 512 contiguous bytes
__device__ __forceinline__ void stage_store_rows16(uint32_t stage, int lane, int half, uint8_t* g, long long pitch, int nch, int nrows) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = 16 * half + 4 * i + (lane >> 3), ch = lane & 7;
    const uint4 v = ld_shared_u4(stage + (uint32_t)row * 128u + ((uint32_t)(ch ^ (row & 7)) << 4));
    if (row < nrows && ch < nch) *reinterpret_cast<uint4*>(g + row * pitch + ch * 16) = v;
  }
}
__device__ __forceinline__ void stage_put_rows16(uint32_t stage, int lane, int half, const uint4 (&v)[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = 16 * half + 4 * i + (lane >> 3), ch = lane & 7;
    st_shared_u4(stage + (uint32_t)row * 128u + ((uint32_t)(ch ^ (row & 7)) << 4), v[i]);
  }
}
// LayerNorm over the n channels of a pixel held by two threads (16 channels each) of different warps: partial sums meet in
// shared memory (xs / xq: one float per (half, tile row)), two pair barriers; biased variance, as nn.LayerNorm
__device__ __forceinline__ void layer_norm_pair(float (&v)[16], int half, int n, const float* gamma, const float* beta, float eps,
                                                float* xs, float* xq, int t, int pair_id) {
  const int c0 = 16 * half;
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) sum += c0 + j < n ? v[j] : 0.f;
  xs[half * TILE_ROWS + t] = sum;
  pair_sync(pair_id);
  const float mean = (sum + xs[(half ^ 1) * TILE_ROWS + t]) / (float)n;
  float sq = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float d = c0 + j < n ? v[j] - mean : 0.f;
    sq = fmaf(d, d, sq);
  }
  xq[half * TILE_ROWS + t] = sq;
  pair_sync(pair_id);
  const float rstd = 1.f / sqrtf((sq + xq[(half ^ 1) * TILE_ROWS + t]) / (float)n + eps);
#pragma unroll
  for (int j = 0; j < 16; j += 4) {
    const float4 g = *reinterpret_cast<const float4*>(gamma + c0 + j);
    const float4 b = *reinterpret_cast<const float4*>(beta + c0 + j);
    if (c0 + j < n) {
      v[j] = (v[j] - mean) * rstd * g.x + b.x;
      v[j + 1] = (v[j + 1] - mean) * rstd * g.y + b.y;
      v[j + 2] = (v[j + 2] - mean) * rstd * g.z + b.z;
      v[j + 3] = (v[j + 3] - mean) * rstd * g.w + b.w;
    }
  }
}

// descriptor of a K-major 128B-swizzled operand tile from its low word (start address >> 4 | LBO): the high word (stride
// 1024 B, version, swizzle mode) is a constant, so K offsets are 32-bit adds and the compiler keeps the high word in one
// uniform register (the MMA issuers are single threads whose instruction stream bounds the kernel, see below)
constexpr uint32_t DESC_HI = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3ffffu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc64(uint32_t lo) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(DESC_HI));
  return d;
}

__global__ void __launch_bounds__(PIX_THREADS, 1)
conv_pix_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w1,
                const __grid_constant__ CUtensorMap tm_w2, const PixArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w1_base = smem_base + (uint32_t)p.stages * A_STAGE;
  const uint32_t w2_base = w1_base + (uint32_t)p.taps * W1_TAP;
  const uint32_t a2_base = w2_base + (p.gated ? W2_BYTES : 0);   // gate operand tile = the epilogue warps' staging blocks
  const uint32_t bar_base = a2_base + A_STAGE;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (MAX_STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * MAX_STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * MAX_STAGES + NBUF + s); };
  const uint32_t wfull_bar = bar_base + 8u * (2 * MAX_STAGES + 2 * NBUF);
  const uint32_t a2full_bar = bar_base + 8u * (2 * MAX_STAGES + 2 * NBUF + 1);
  const uint32_t acc2full_bar = bar_base + 8u * (2 * MAX_STAGES + 2 * NBUF + 2);
  const uint32_t tmem_slot = bar_base + 8u * (2 * MAX_STAGES + 2 * NBUF + 3);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  // per-channel constants of the epilogue (bias1[32] | bias2[64] | gamma[32] | beta[32]): broadcast shared-memory reads
  // instead of ~200 uniform global loads per pixel thread and tile
  float* s_par = reinterpret_cast<float*>(smem_raw + (bar_base + 256u - smem_u32(smem_raw)));
  float* s_xs = s_par + 192;                           // LayerNorm partial sums / squares of the two column halves: 2 x 2 x 256 floats
  float* s_xq = s_xs + 2 * TILE_ROWS;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_chains = (p.taps + p.chain_taps - 1) / p.chain_taps;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_w1);
    if (p.gated) prefetch_tmap(&tm_w2);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), MT); }
      for (int s = 0; s < NBUF; ++s) { mbar_init(tfull_bar(s), MT); mbar_init(tempty_bar(s), PIX_EPI_WARPS); }
      mbar_init(wfull_bar, 1);
      mbar_init(a2full_bar, PIX_EPI_WARPS);
      mbar_init(acc2full_bar, MT);
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // Programmatic dependent launch (common.cuh): everything above touches only kernel parameters and this CTA's shared /
  // tensor memory, so it may run while the previous kernel of the chain drains; every thread that reads or writes global
  // memory (the producer -- weights included: they may come from the kernel just before --, the epilogue warps) waits first.
  griddep_launch_dependents();

  // What the measurements decided (DESIGN.md 4.3, profiles/r02_conv_pix_probe.log):
  //  * no setmaxnreg (640 threads x 96 registers; the 56 / 224 split of the flat kernels made the issuer re-load its
  //    descriptors from local memory in front of every tcgen05.mma; and setmaxnreg.inc can only take what .dec released
  //    inside the CTA's launch allocation);
  //  * the issuing threads are chosen with elect.sync, not `lane == 0`: the compiler then emits tcgen05.mma / TMA back to
  //    back instead of wrapping each one in an ELECT / BRA.U.ANY loop that waits for the instruction's scoreboard;
  //  * ONE thread per role runs the barrier protocol (32 lanes polling an mbarrier serialise), and a wait first tries the
  //    non-blocking test_wait (16 cycles on a completed phase against ~180 for try_wait);
  //  * the issuer's own instruction stream (~20 instructions per MMA of 16-44 tensor cycles at N = 32) is what bounds the
  //    kernel, so each of the two 128-row MMA tiles of a CTA tile has its own issuer warp.
  if (warp < FIRST_EPI_WARP) {
    if (warp == 0) {
      // ===================== TMA producer: the weights once, then one box per (tile, tap) =====================
      if (elect_one()) {
        griddep_wait();
        mbar_expect_tx(wfull_bar, (uint32_t)p.taps * W1_TAP + (p.gated ? W2_BYTES : 0));
        for (int tap = 0; tap < p.taps; ++tap) tma_load_2d(w1_base + (uint32_t)tap * W1_TAP, &tm_w1, wfull_bar, tap * 64, 0);
        if (p.gated) tma_load_2d(w2_base, &tm_w2, wfull_bar, 0, 0);
        const int half = p.ksize >> 1;
        int stage = 0;
        uint32_t phase = 0;
        for (long long tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
          const Tile t = decode_tile(p, tile);
          for (int ty = 0; ty < p.ksize; ++ty)
            for (int tx = 0; tx < p.ksize; ++tx) {
              mbar_wait(empty_bar(stage), phase ^ 1);
              mbar_expect_tx(full_bar(stage), p.box_bytes);
              tma_load_4d(smem_base + (uint32_t)stage * A_STAGE, &tm_a, full_bar(stage), 0, (tx - half) * p.dil,
                          t.h0 + (ty - half) * p.dil, t.n0);
              if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
      }
    } else if (warp <= MT && elect_one()) {
      // ===================== MMA issuers: warp 1 + mt issues every product of MMA tile mt =====================
      const int mt = warp - 1;
      mbar_wait(wfull_bar, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0, a2_phase = 0;
      bool pending = false;                              // the previous tile's 1 x 1 contraction has not been issued yet
      const int gate_max = n_chains > NBUF ? NBUF : n_chains - 1;
      const int gate_at = p.gate_at < gate_max ? p.gate_at : gate_max;
      const uint32_t a_lo0 = desc_lo(smem_base + (uint32_t)mt * A_MT), w_lo0 = desc_lo(w1_base);
      const uint32_t d_col = tmem_base + (uint32_t)mt * 32;
      auto gate_mma = [&]() {
        mbar_wait(a2full_bar, a2_phase);
        a2_phase ^= 1;
        tcgen05_fence_after();
        const uint32_t da = desc_lo(a2_base + (uint32_t)mt * A_MT), db = desc_lo(w2_base);
        const uint32_t d = tmem_base + ACC2_COL + (uint32_t)mt * 64;
        umma_f16(desc64(da + KOFF_LO), desc64(db), d, IDESC_N64, 0u);
        umma_f16(desc64(da), desc64(db + KOFF_LO), d, IDESC_N64, 1u);
        umma_f16(desc64(da + KOFF_LO + KOFF_K1), desc64(db + KOFF_K1), d, IDESC_N64, 1u);
        umma_f16(desc64(da + KOFF_K1), desc64(db + KOFF_LO + KOFF_K1), d, IDESC_N64, 1u);
        umma_f16_scale11(desc64(da), desc64(db), d, IDESC_N64);
        umma_f16(desc64(da + KOFF_K1), desc64(db + KOFF_K1), d, IDESC_N64, 1u);
        umma_commit(acc2full_bar);
      };
      for (long long tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        for (int c = 0; c < n_chains; ++c) {
          // the gate contraction of the PREVIOUS tile goes behind this tile's chains (in front of the last one): the tensor
          // pipe has them to work on while the epilogue warps build that operand tile.  Never behind more than NBUF chains:
          // chain NBUF needs the accumulator of chain 0 drained, and the epilogue warps drain it only after they have
          // consumed the gate accumulator.
          if (pending && c == gate_at) { gate_mma(); pending = false; }
          const int tap0 = c * p.chain_taps;
          const int tap1 = tap0 + p.chain_taps < p.taps ? tap0 + p.chain_taps : p.taps;
          mbar_wait(tempty_bar(acc), acc_phase ^ 1);
          tcgen05_fence_after();
          const uint32_t d = d_col + (uint32_t)acc * 64;
          int st = stage;
          uint32_t ph = phase;
          for (int tap = tap0; tap < tap1; ++tap) {       // cross terms of the whole chain first (lo' is scaled by 2^11)
            mbar_wait(full_bar(st), ph);
            const uint32_t da = a_lo0 + (uint32_t)st * (A_STAGE >> 4), db = w_lo0 + (uint32_t)tap * (W1_TAP >> 4);
            umma_f16(desc64(da + KOFF_LO), desc64(db), d, IDESC_N32, tap > tap0 ? 1u : 0u);
            umma_f16(desc64(da), desc64(db + KOFF_LO), d, IDESC_N32, 1u);
            umma_f16(desc64(da + KOFF_LO + KOFF_K1), desc64(db + KOFF_K1), d, IDESC_N32, 1u);
            umma_f16(desc64(da + KOFF_K1), desc64(db + KOFF_LO + KOFF_K1), d, IDESC_N32, 1u);
            if (++st == p.stages) { st = 0; ph ^= 1; }
          }
          for (int tap = tap0; tap < tap1; ++tap) {       // hi.hi: the first one rescales the accumulator by 2^-11
            const uint32_t da = a_lo0 + (uint32_t)stage * (A_STAGE >> 4), db = w_lo0 + (uint32_t)tap * (W1_TAP >> 4);
            if (tap == tap0) umma_f16_scale11(desc64(da), desc64(db), d, IDESC_N32);
            else umma_f16(desc64(da), desc64(db), d, IDESC_N32, 1u);
            umma_f16(desc64(da + KOFF_K1), desc64(db + KOFF_K1), d, IDESC_N32, 1u);
            umma_commit(empty_bar(stage));
            if (tap == tap1 - 1) umma_commit(tfull_bar(acc));
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          if (++acc == NBUF) { acc = 0; acc_phase ^= 1; }
        }
        pending = p.gated != 0;
      }
      if (pending) gate_mma();
    }
  } else {
    // ===================== epilogue warps: two threads (of two warps) per pixel, 16 channels each =====================
    // (one thread per pixel with all 32 channels was ~2 600 instructions per tile on two warps per scheduler and bound the
    //  gated block; the pair meets in shared memory for the LayerNorm statistics and shares the 32-row staging block)
    const int e = warp - FIRST_EPI_WARP;
    const int q = e & 3, mt = (e >> 2) & 1, half = e >> 3;
    const int pair_id = 1 + (e & 7);                                  // named barrier of the two warps of a block
    const int c0 = 16 * half;                                         // first channel of this thread
    const int wrow0 = mt * BLOCK_M + q * 32;                          // first tile row of the pair's block
    const int t = wrow0 + lane;                                       // row of the CTA tile
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t stage = a2_base + (uint32_t)wrow0 * 128u;          // the pair's 4 KB block (rows wrow0 .. wrow0 + 31)
    const bool x_vec = p.x && p.c_x % 4 == 0 && p.ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(p.x) & 15) == 0;
    int acc = 0;
    uint32_t acc_phase = 0, acc2_phase = 0;
    griddep_wait();
    {                                                    // per-channel constants -> shared memory (the 512 epilogue threads)
      const int i = threadIdx.x - FIRST_EPI_WARP * 32;
      if (i < 160) {
        float v = 0.f;
        if (i < 32) v = p.bias1[i];
        else if (i < 96) v = p.gated ? p.bias2[i - 32] : 0.f;
        else if (i < 128) v = (p.gamma && i - 96 < p.n1) ? p.gamma[i - 96] : 0.f;
        else v = (p.beta && i - 128 < p.n1) ? p.beta[i - 128] : 0.f;
        s_par[i] = v;
      }
      asm volatile("bar.sync 9, %0;" ::"n"(PIX_EPI_WARPS * 32) : "memory");
    }
    // The rows a tile's epilogue READS (gated: the residual stream; last convolution: x) are fetched ONE TILE AHEAD, as soon
    // as the previous tile has moved its copy into the staging block (this warp: 16 of the block's 32 rows, 512 contiguous
    // bytes per instruction): issued at the top of their own tile they queued behind the previous tile's stores and their
    // latency showed (the gated block: 166 -> 15x us).
    uint4 pre[4];
    const bool pre_on = p.gated || x_vec;
    const uint8_t* pre_base = p.gated ? reinterpret_cast<const uint8_t*>(p.out_f32) : reinterpret_cast<const uint8_t*>(p.x);
    const long long pre_pitch = p.gated ? p.ld_f32 * 4 : p.ldx * 4;
    const int pre_nch = p.gated ? 8 : (p.c_x >> 2);
    auto prefetch = [&](long long tile_) {
      if (!pre_on || tile_ >= p.n_tiles) return;
      const Tile tn = decode_tile(p, tile_);
      int rows_ = tn.nvalid - wrow0;
      rows_ = rows_ < 0 ? 0 : rows_ > 32 ? 32 : rows_;
      const uint8_t* g_ = pre_base + (tn.row0 + wrow0) * pre_pitch;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = 16 * half + 4 * i + (lane >> 3), ch = lane & 7;
        pre[i] = make_uint4(0u, 0u, 0u, 0u);
        if (row < rows_ && ch < pre_nch) pre[i] = *reinterpret_cast<const uint4*>(g_ + row * pre_pitch + ch * 16);
      }
    };
#pragma unroll
    for (int i = 0; i < 4; ++i) pre[i] = make_uint4(0u, 0u, 0u, 0u);
    prefetch(blockIdx.x);
    for (long long tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      const Tile tl = decode_tile(p, tile);
      const bool valid = t < tl.nvalid;
      int wrows = tl.nvalid - wrow0;                                  // valid rows of the pair's block
      wrows = wrows < 0 ? 0 : wrows > 32 ? 32 : wrows;
      const long long r = tl.row0 + t, wr = tl.row0 + wrow0;
      float m[16];
      for (int c = 0; c < n_chains; ++c) {
        if (lane == 0) mbar_wait(tfull_bar(acc), acc_phase);
        __syncwarp();
        tcgen05_fence_after();
        float v[16];
        tmem_ld16(lane_addr + acc * 64 + mt * 32 + c0, v);
        tmem_ld_wait();
        if (c == 0) {
#pragma unroll
          for (int j = 0; j < 16; ++j) m[j] = v[j];
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) m[j] += v[j];
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
        if (++acc == NBUF) { acc = 0; acc_phase ^= 1; }
      }
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const float4 b = *reinterpret_cast<const float4*>(s_par + c0 + j);
        m[j] += b.x; m[j + 1] += b.y; m[j + 2] += b.z; m[j + 3] += b.w;
      }
      if (!p.gated) {
        if (p.relu1) {
#pragma unroll
          for (int j = 0; j < 16; ++j) m[j] = fmaxf(m[j], 0.f);
        }
        if (p.gamma) layer_norm_pair(m, half, p.n1, s_par + 96, s_par + 128, p.eps, s_xs, s_xq, t, pair_id);
        if (p.x) {                                                    // x[r, c] += sign * (1 - mask)[pixel, c] * v[c]
          const int pix = (tl.h0 * p.W + t) % p.HW;
          const float* g = p.inv_mask + (long long)pix * p.c_x;
          if (x_vec) {
            uint8_t* xg = reinterpret_cast<uint8_t*>(p.x + wr * p.ldx);
            stage_put_rows16(stage, lane, half, pre);
            pair_sync(pair_id);
            prefetch(tile + gridDim.x);
            float xr[16];
            stage_read_f32_half(stage, lane, half, xr);
            if (valid) {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (c0 + j < p.c_x) xr[j] = fmaf(p.sign * __ldg(g + c0 + j), m[j], xr[j]);
            }
            stage_write_f32_half(stage, lane, half, xr);            // (own chunks only: read and written by this thread)
            pair_sync(pair_id);
            stage_store_rows16(stage, lane, half, xg, p.ldx * 4, p.c_x >> 2, wrows);
            pair_sync(pair_id);
          } else if (valid) {
            float* xr = p.x + r * p.ldx;
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + j < p.c_x) xr[c0 + j] = fmaf(p.sign * __ldg(g + c0 + j), m[j], xr[c0 + j]);
          }
        }
        if (p.out_f32) {
          stage_write_f32_half(stage, lane, half, m);
          pair_sync(pair_id);
          stage_store_rows16(stage, lane, half, reinterpret_cast<uint8_t*>(p.out_f32 + wr * p.ld_f32), p.ld_f32 * 4, p.n1 >> 2, wrows);
          pair_sync(pair_id);
        }
        if (p.out16) {
          const bool bad = p.relu_planes ? stage_write_planes_half<true>(stage, lane, half, m)
                                         : stage_write_planes_half<false>(stage, lane, half, m);
          if (bad && valid && p.overflow_flag) *p.overflow_flag = 1;
          pair_sync(pair_id);
          stage_store_rows16(stage, lane, half, reinterpret_cast<uint8_t*>(p.out16) + wr * PIX_BYTES, PIX_BYTES, 8, wrows);
          pair_sync(pair_id);
        }
      } else {
        // the residual stream's rows of this block, through the staging block (free: the previous tile's stores ended with
        // a pair barrier, its gate contraction has been consumed)
        uint8_t* yg = reinterpret_cast<uint8_t*>(p.out_f32 + wr * p.ld_f32);
        float y[16];
        stage_put_rows16(stage, lane, half, pre);
        pair_sync(pair_id);
        stage_read_f32_half(stage, lane, half, y);
        pair_sync(pair_id);                              // both halves have read their channels: the block becomes the operand
        // u = relu(conv + b) -> the pair's rows of the operand tile of the 1 x 1 convolution (= its staging block)
        if (!valid) {                                    // rows past the tile's pixels: a zero operand row
#pragma unroll
          for (int j = 0; j < 16; ++j) m[j] = 0.f;
        }
        const bool bad = stage_write_planes_half<true>(stage, lane, half, m);
        if (bad && p.overflow_flag) *p.overflow_flag = 1;
        fence_proxy_async_smem();
        tcgen05_fence_before();                          // (our reads of the gate accumulator for the previous tile are done)
        __syncwarp();
        if (lane == 0) mbar_arrive(a2full_bar);
        prefetch(tile + gridDim.x);                      // (its registers were emptied into the staging block above)
        if (lane == 0) mbar_wait(acc2full_bar, acc2_phase);
        __syncwarp();
        acc2_phase ^= 1;
        tcgen05_fence_after();
        {
          // sigmoid with ex2.approx / rcp.approx (a few ulp)
          float g[16];
          tmem_ld16(lane_addr + ACC2_COL + mt * 64 + 32 + c0, g);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 b = *reinterpret_cast<const float4*>(s_par + 64 + c0 + j);
            m[j] = __fdividef(1.f, 1.f + __expf(-(g[j] + b.x)));
            m[j + 1] = __fdividef(1.f, 1.f + __expf(-(g[j + 1] + b.y)));
            m[j + 2] = __fdividef(1.f, 1.f + __expf(-(g[j + 2] + b.z)));
            m[j + 3] = __fdividef(1.f, 1.f + __expf(-(g[j + 3] + b.w)));
          }
          tmem_ld16(lane_addr + ACC2_COL + mt * 64 + c0, g);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 b = *reinterpret_cast<const float4*>(s_par + 32 + c0 + j);
            y[j] = fmaf(g[j] + b.x, m[j], y[j]);
            y[j + 1] = fmaf(g[j + 1] + b.y, m[j + 1], y[j + 1]);
            y[j + 2] = fmaf(g[j + 2] + b.z, m[j + 2], y[j + 2]);
            y[j + 3] = fmaf(g[j + 3] + b.w, m[j + 3], y[j + 3]);
          }
        }
        tcgen05_fence_before();
        if (p.post_relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) y[j] = fmaxf(y[j], 0.f);
        }
        if (p.gamma) layer_norm_pair(y, half, p.n1, s_par + 96, s_par + 128, p.eps, s_xs, s_xq, t, pair_id);
        // (the gate contraction has completed -- acc2full, observed by BOTH warps before the pair barriers of the LayerNorm
        //  or the one below -- so the tensor core is done reading the staging block)
        if (!p.gamma) pair_sync(pair_id);
        stage_write_f32_half(stage, lane, half, y);
        pair_sync(pair_id);
        stage_store_rows16(stage, lane, half, yg, p.ld_f32 * 4, 8, wrows);
        pair_sync(pair_id);
        if (p.out16) {
          const bool bad2 = p.relu_planes ? stage_write_planes_half<true>(stage, lane, half, y)
                                          : stage_write_planes_half<false>(stage, lane, half, y);
          if (bad2 && valid && p.overflow_flag) *p.overflow_flag = 1;
          pair_sync(pair_id);
          stage_store_rows16(stage, lane, half, reinterpret_cast<uint8_t*>(p.out16) + wr * PIX_BYTES, PIX_BYTES, 8, wrows);
          pair_sync(pair_id);
        }
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}

// fp32 channels-last rows [rows, C] (C <= 32) -> pixel planes, fused with the coupling's x * mask and an optional ReLU.
// One thread per (pixel, 8-channel chunk).
__global__ void __launch_bounds__(256)
pix_encode_kernel(const float* __restrict__ x, long long ldx, long long rows, int C, int HW, const float* __restrict__ mask,
                  int relu, __half* __restrict__ out16, int* overflow_flag) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * 4) return;
  const long long r = idx >> 2;
  const int c = (int)(idx & 3);
  float v[8];
  const float* xr = x + r * ldx;
  const float* mr = mask ? mask + (long long)(r % HW) * C : nullptr;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = 8 * c + i;
    float t = ch < C ? xr[ch] : 0.f;
    if (mr && ch < C) t *= __ldg(mr + ch);
    v[i] = relu ? fmaxf(t, 0.f) : t;
  }
  uint4 hi, lo;
  const bool bad = split8(v, hi, lo);
  uint8_t* dst = reinterpret_cast<uint8_t*>(out16) + r * PIX_BYTES;
  *reinterpret_cast<uint4*>(dst + 16 * c) = hi;
  *reinterpret_cast<uint4*>(dst + 64 + 16 * c) = lo;
  if (bad && overflow_flag) *overflow_flag = 1;
}

}  // namespace convpix

// host side -----------------------------------------------------------------------------------------------
// tile geometry of usf_conv2d_pix for an H x W image; false when the image does not fit the 256-row tile scheme
inline bool conv_pix_geometry(int H, int W, int* imgs, int* hr, int* tiles_per_img) {
  const int HW = H * W;
  if (W > 256) return false;
  if (HW <= convpix::TILE_ROWS) {
    *imgs = convpix::TILE_ROWS / HW;
    if (*imgs > 256) *imgs = 256;
    *hr = H;
    *tiles_per_img = 1;
  } else {
    *imgs = 1;
    *hr = convpix::TILE_ROWS / W;
    *tiles_per_img = (H + *hr - 1) / *hr;
  }
  return true;
}
// pipeline stages that fit next to the resident weights (0: the shape does not fit)
inline int conv_pix_stages(int taps, int gated) {
  const long long fixed = (long long)taps * convpix::W1_TAP + (gated ? convpix::W2_BYTES : 0) + convpix::A_STAGE + 1024 + 6144;
  long long s = (227 * 1024 - fixed) / convpix::A_STAGE;
  if (s > convpix::MAX_STAGES) s = convpix::MAX_STAGES;
  return s >= 2 ? (int)s : 0;
}
inline size_t conv_pix_smem_bytes(int taps, int gated) {
  return (size_t)conv_pix_stages(taps, gated) * convpix::A_STAGE + (size_t)taps * convpix::W1_TAP +
         (gated ? convpix::W2_BYTES : 0) + convpix::A_STAGE + 1024 + 6144;
}

int launch_conv_pix(const usf_conv_pix_args* a, cudaStream_t st);
int launch_pix_encode(const float* x, long long ldx, long long rows, int c, int hw, const float* mask, int relu, void* out16,
                      int* overflow_flag, cudaStream_t st);

}  // namespace usf
