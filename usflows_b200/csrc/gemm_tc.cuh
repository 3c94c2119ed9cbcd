// Shared tcgen05 / TMEM / TMA primitives for sm_100a, and the single-CTA pieces of the implicit-GEMM convolution
// (conv_tc.cuh).  The contraction itself is the CTA-pair kernel of gemm_tc2.cuh.
//
//   * mbarrier, elect, fence, TMA load, tcgen05.mma / commit and tcgen05.ld helpers used by every tcgen05 kernel
//     (gemm_tc2.cuh, conv_tc.cuh, conv_pix.cuh)
//   * operands K-major in shared memory, 128-byte swizzle, one 128 B K-slab per pipeline stage (32 tf32/fp32 elements
//     or 64 bf16/fp16 elements): make_operand_map builds the TMA map (hardware zero fill for the M / N / K tails),
//     make_smem_desc the matching shared-memory descriptor
//   * warp roles of the warp-specialised kernels: warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 4..11
//     epilogue (warp w owns TMEM lane quarter w % 4 and one half of the tile's columns); the epilogue warpgroups take
//     the register file with setmaxnreg
//   * tc::Config + epilogue_loop: the single-CTA (cta_group::1, M = 128) tile and its epilogue warps.  The tensor core
//     adds into its fp32 accumulator with truncation, so a long K chain carries a systematic toward-zero bias (~0.2 ulp
//     per MMA step, measured: 5e-6 relative at K=1024 x 3 terms, coherent across layers); the fp32-accurate mode
//     therefore closes the TMEM accumulator every `chunk_slabs` K-slabs and the epilogue warps add the partial tile into
//     fp32 registers with round-to-nearest (two TMEM accumulators ping-pong between the MMA issuer and the epilogue)
#pragma once
#include "common.cuh"

namespace usf {

#ifndef USF_WATCHDOG
#define USF_WATCHDOG 1
#endif

namespace tc {

constexpr int BLOCK_M = 128;
constexpr int SLAB_BYTES = 128;  // K extent of one stage in bytes (= swizzle span)
constexpr int UMMA_K_BYTES = 32;
constexpr int NUM_THREADS = 384;   // warpgroup 0: TMA producer, MMA issuer, 2 idle warps; warpgroups 1-2: epilogue
constexpr int NUM_EPI_WARPS = 8;
constexpr int FIRST_EPI_WARP = 4;
constexpr int REGS_NON_EPI = 56;   // setmaxnreg budget after role dispatch: 128*56 + 256*224 = 64512 (<= 65536 with slack; an exact fit can block setmaxnreg.inc forever)
constexpr int REGS_EPI = 224;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  // fast path: the non-blocking test costs ~16 cycles on a completed phase, the (potentially suspending) try_wait ~180
  // even when the phase is already complete (measured in-kernel on a B200) -- and in a full pipeline most
  // waits find their phase complete
  if (mbar_test_wait(bar, parity)) return;
#if USF_WATCHDOG
  unsigned long long t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) {  // 4 s: a protocol bug, not a slow tile -> abort the launch
        printf("usflows_b200: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n",
               (int)blockIdx.x, (int)threadIdx.x, bar, parity);
        __trap();
      }
    }
  }
#else
  while (!mbar_try_wait(bar, parity)) {}
#endif
}

// one thread of the (converged) warp: elect.sync tells the compiler the branch is taken by exactly one lane, so the
// uniform-datapath instructions inside (tcgen05.mma, tcgen05.commit, TMA) need no per-lane ELECT / BRA.U.ANY loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// K-major, 128B-swizzled operand tile: rows at a 128 B pitch, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3ffff) >> 4);  // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset = 8 rows * 128 B
  d |= (uint64_t)1 << 46;                        // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}

template <bool BF16>
__device__ __forceinline__ void umma(uint64_t da, uint64_t db, uint32_t tmem_d, uint32_t idesc, uint32_t accumulate) {
  if (BF16) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// single-CTA (cta_group::1, M = 128) tile: TMEM accumulator layout, epilogue column halves, instruction descriptor
template <int BLOCK_N, int NTERMS, bool BF16>
struct Config {
  static_assert(BLOCK_N % 16 == 0 && BLOCK_N >= 16 && BLOCK_N <= 256, "UMMA N for M=128");
  static_assert(NTERMS == 1 || NTERMS == 3, "1 = single pass, 3 = tf32 split");
  static constexpr int kBlockN = BLOCK_N;
  static constexpr int ACC_STRIDE = BLOCK_N <= 32 ? 32 : BLOCK_N <= 64 ? 64 : BLOCK_N <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;  // power of two >= 64
  static constexpr int HALF0 = ((BLOCK_N / 16 + 1) / 2) * 16;  // columns owned by epilogue warps 4..7
  static constexpr int HALF1 = BLOCK_N - HALF0;                // ... and by warps 8..11 (may be 0)
  // instruction descriptor: D=f32, A/B = tf32 (2) or bf16 (1), both K-major, N>>3, M>>4
  static constexpr uint32_t IDESC = (1u << 4) | ((BF16 ? 1u : 2u) << 7) | ((BF16 ? 1u : 2u) << 10) |
                                    ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
};

// One epilogue warp: owns TMEM lanes [32*quarter, 32*quarter+32) and columns [col0, col0+COLS) of every tile.
// Partial accumulators (one per K chunk) are summed in fp32 registers (round-to-nearest), then the fused
// epilogue runs on the register tile.  tfull0/tempty0 are the addresses of barrier 0 of each pair (8 B apart).
template <class C, int COLS>
__device__ __forceinline__ void epilogue_loop(int col0, int quarter, int lane, uint32_t tmem_base, uint32_t tfull0,
                                              uint32_t tempty0, long long n_tiles, int n_blocks, int k_slabs,
                                              int chunk_slabs, long long M, int N, const Epilogue& ep) {
  constexpr int BLOCK_N = C::kBlockN;
  int acc = 0;
  uint32_t acc_phase = 0;
  const int n_chunks = (k_slabs + chunk_slabs - 1) / chunk_slabs;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long m_idx = (tile / n_blocks) * BLOCK_M;
    const int n_idx = (int)(tile % n_blocks) * BLOCK_N;
    const long long row = m_idx + quarter * 32 + lane;
    if (COLS == 0) {  // nothing to own (BLOCK_N == 16): still take part in the barrier protocol
      for (int c = 0; c < n_chunks; ++c) {
        mbar_wait(tfull0 + 8u * acc, acc_phase);
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty0 + 8u * acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      continue;
    }
    float master[COLS > 0 ? COLS : 1];
    for (int c = 0; c < n_chunks; ++c) {
      mbar_wait(tfull0 + 8u * acc, acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * C::ACC_STRIDE + col0;
#pragma unroll
      for (int j = 0; j < COLS; j += 16) {
        float v[16];
        tmem_ld16(taddr + j, v);
        tmem_ld_wait();
        if (c == 0) {
#pragma unroll
          for (int i = 0; i < 16; ++i) master[j + i] = v[i];
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) master[j + i] += v[i];
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8u * acc);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (row < M) {
#pragma unroll
      for (int j = 0; j < COLS; j += 16) {
        if (n_idx + col0 + j < N)
          epi_row_chunk<16>(ep, *reinterpret_cast<float(*)[16]>(&master[j]), row, n_idx + col0 + j, N);
      }
    }
  }
}

}  // namespace tc

// host side ---------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();

// 2-D row-major [rows, cols] operand, box = 128 B of K x box_rows rows, 128B swizzle, zero OOB fill
// dtype: 0 = fp32 / tf32, 1 = bf16, 2 = fp16
inline int make_operand_map(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld,
                            int box_rows, int dtype) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return fail(USF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available%s%s");
  const int esz = dtype ? 2 : 4;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)(tc::SLAB_BYTES / esz), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, dtype == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : dtype == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)",
             (int)r, rows, cols, ld);
    return USF_ERR_CUDA;
  }
  return USF_OK;
}

}  // namespace usf
