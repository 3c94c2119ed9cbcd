// tcgen05 contraction, CTA-pair version (cta_group::2):  out = epilogue( sum_terms A_t[M,K] . W_t[N,K]^T )
//
// Two CTAs of a cluster (one TPC) share every MMA: UMMA M = 256 (128 rows of A per CTA), N = BLOCK_N with
// each CTA staging only HALF of the W tile, so the shared-memory fill traffic per MMA cycle drops by a third
// against a single-CTA (M = 128) tile -- a single-CTA contraction is bound by the L2 -> SM fill rate
// (~40 B/cycle/SM measured), not by the tensor pipe.
//
//   * per CTA and K-slab (128 B of K): A tile 128 rows + W half tile BLOCK_N/2 rows, per operand plane,
//     K-major, 128B swizzle, filled by TMA (cp.async.bulk.tensor.2d.cta_group::2); both CTAs' loads complete
//     on the LEADER's full barrier (armed with the byte count of both)
//   * the leader's MMA thread issues tcgen05.mma.cta_group::2; tcgen05.commit multicasts the "slot free" and
//     "accumulator ready" arrivals to both CTAs; each CTA's epilogue drains its own 128 TMEM lanes and
//     releases the accumulator on the leader's barrier (remote mbarrier.arrive)
//   * fp32 mode (NTERMS = 3): the accumulation chain is closed every `chunk_slabs` K-slabs and promoted into
//     fp32 registers with round-to-nearest (the tensor core accumulates with truncation, see gemm_tc.cuh); two TMEM
//     accumulators ping-pong
//   * epilogue: registers -> per-warp padded smem patch (16 columns at a time) -> coalesced 64 B row segments
//     with the fused bias / ReLU / residual / column scale / post-subtract / hi-lo or bf16 re-encoding
#pragma once
#include "gemm_tc.cuh"

namespace usf {
namespace tc2 {

using namespace tc;  // mbarrier / TMA / descriptor / TMEM helpers

constexpr int PATCH_COLS = 16;                 // epilogue staging granularity
constexpr int PATCH_LD = PATCH_COLS + 4;       // padded row pitch (floats): conflict-free v4 writes and reads
constexpr int PATCH_BYTES = 32 * PATCH_LD * 4; // one warp: 32 rows

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t num_clusters_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory offset in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// remote arrive.  No cluster-scope release: the only thing handed over is TMEM ownership, which is ordered by the
// tcgen05 fences; a .release.cluster arrive compiles to a full ERRBAR fence per call (22% of all stall samples
// of the first version of this kernel, profiles/r01_full_gemm_v2_fp32.md)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
constexpr int STAGE_EPI_BYTES = 4096;          // per epilogue warp: one 32-row x (128 B | 2 x 64 B) staging box
constexpr int INBOX_BYTES = 2048;              // per epilogue warp: one plane of a 32-row x 32-column residual piece

// Accumulation-chain schedule of one tile: the first `lead` chains span 2 * chunk K-slabs, the others `chunk`.
// Longer leading chains let the MMA issuer run further ahead while the epilogue warps are still storing the previous
// tile (two TMEM accumulators = two chains of run-ahead); they cost a little accumulation accuracy (longer chains).
__device__ __forceinline__ int chain_lead(int k_slabs, int chunk, int lead) {
  const int fit = k_slabs / (2 * chunk);
  return lead < fit ? lead : fit;
}
__device__ __forceinline__ int chain_count(int k_slabs, int chunk, int lead) {
  const int l = chain_lead(k_slabs, chunk, lead);
  return l + (k_slabs - 2 * chunk * l + chunk - 1) / chunk;
}

// Work item of the persistent loop: output tile (m_blk, n_blk) x K range [ks_begin, ks_begin + nks) in K-slabs.  With
// split_k > 1 (dW = dY^T . X of the training pass: a small output and a contraction over all batch rows) the K range of a
// tile is cut into split_k pieces that run on different CTA pairs and meet in the fp32 output through red.global.add.
struct TileCoord { long long m_blk; int n_blk; int ks_begin; int nks; };
template <bool SPLITK>
__device__ __forceinline__ TileCoord decode_tile(long long tile, int n_blocks, int split_k, int k_slabs, int per) {
  TileCoord t;
  if (!SPLITK) {
    t.m_blk = tile / n_blocks;
    t.n_blk = (int)(tile % n_blocks);
    t.ks_begin = 0;
    t.nks = k_slabs;
    return t;
  }
  const int sk = (int)(tile % split_k);
  const long long mn = tile / split_k;
  t.m_blk = mn / n_blocks;
  t.n_blk = (int)(mn % n_blocks);
  t.ks_begin = sk * per;               // `per` = K-slabs per piece (a whole number of accumulation chains; the launcher's)
  const int rest = k_slabs - t.ks_begin;
  t.nks = rest < per ? rest : per;     // > 0: the launcher keeps (split_k - 1) * per < k_slabs
  return t;
}

constexpr int KIND_TF32 = 0, KIND_BF16 = 1, KIND_F16 = 2;   // KIND_F16: fp16 split planes (x = hi + lo' 2^-11)

// D = A.B + D * 2^-11 (kind::f16 with scale-input-d): folds the scaled-up cross terms of the fp16 split into the
// accumulator at the moment the first hi.hi product arrives
__device__ __forceinline__ void umma_pair_f16_scale11(uint64_t da, uint64_t db, uint32_t tmem_d, uint32_t idesc) {
  const uint32_t z = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p, 11;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(1u), "r"(z)
      : "memory");
}

template <int KIND>
__device__ __forceinline__ void umma_pair(uint64_t da, uint64_t db, uint32_t tmem_d, uint32_t idesc, uint32_t accumulate) {
  if (KIND != KIND_TF32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// arrive (once the MMAs issued so far have retired) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}

// One pipeline stage holds one 128-byte K-slab per operand row (tc::SLAB_BYTES).  Six half-size stages (64-byte rows, 64B
// swizzle) were measured slower on a B200 (784 x 784 over 65 536 rows: 274 vs 246 us; DESIGN.md section 4.2): twice the TMA
// operations per K cost more than the deeper pipeline gives.
template <int BLOCK_N, int NTERMS, int KIND>
struct Config {
  static_assert(BLOCK_N % 16 == 0 && BLOCK_N >= 32 && BLOCK_N <= 256, "UMMA N for M=256 (cta_group::2)");
  static_assert(NTERMS == 1 || NTERMS == 3, "1 = single pass, 3 = tf32 split");
  static constexpr int kBlockN = BLOCK_N;
  static constexpr int HALF_N = BLOCK_N / 2;                 // W rows staged by each CTA (multiple of 8)
  static constexpr int NPLANES = NTERMS == 3 ? 2 : 1;
  static constexpr int A_TILE = BLOCK_M * SLAB_BYTES;        // 16 KB
  static constexpr int B_TILE = HALF_N * SLAB_BYTES;         // multiple of 1024
  static constexpr int STAGE_BYTES = NPLANES * (A_TILE + B_TILE);
  static_assert(PATCH_BYTES <= STAGE_EPI_BYTES, "patch buffer lives in the staging area");
  // a 2 KB "in-box" per epilogue warp (coalesced loads of the coupling residual, see coop_resid_row) where it does not cost
  // a pipeline stage: BLOCK_N = 208 and narrower on the fp16-split engine
  static constexpr int STAGES_PLAIN = (227 * 1024 - 1024 - 512 - NUM_EPI_WARPS * STAGE_EPI_BYTES) / STAGE_BYTES;
  static constexpr int STAGES_INBOX = (227 * 1024 - 1024 - 512 - NUM_EPI_WARPS * (STAGE_EPI_BYTES + INBOX_BYTES)) / STAGE_BYTES;
  static constexpr bool INBOX = KIND == KIND_F16 && NTERMS == 3 &&
                                (STAGES_INBOX >= 8 || STAGES_INBOX == STAGES_PLAIN);
  static constexpr int EPI_BYTES = NUM_EPI_WARPS * (STAGE_EPI_BYTES + (INBOX ? INBOX_BYTES : 0));
  static constexpr int STAGES_RAW = (227 * 1024 - 1024 - 512 - EPI_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static_assert(STAGES >= 2, "need at least a double-buffered pipeline");
  static constexpr int ACC_STRIDE = BLOCK_N <= 32 ? 32 : BLOCK_N <= 64 ? 64 : BLOCK_N <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 1024 /*align slack*/ + 512 /*barriers*/;
  static constexpr int ELEMS_PER_SLAB = SLAB_BYTES / (KIND == KIND_TF32 ? 4 : 2);
  static constexpr uint32_t FMT = KIND == KIND_TF32 ? 2u : KIND == KIND_BF16 ? 1u : 0u;   // idesc operand format
  static constexpr int HALF0 = ((BLOCK_N / 16 + 1) / 2) * 16;  // columns owned by epilogue warps 4..7
  static constexpr int HALF1 = BLOCK_N - HALF0;                // ... and by warps 8..11
  static constexpr uint32_t IDESC_NO_N = (1u << 4) | (FMT << 7) | (FMT << 10) | ((uint32_t)(256 >> 4) << 24);
  // instruction descriptor: D=f32, A/B = tf32 (2), bf16 (1) or f16 (0), both K-major, N>>3, M>>4 with M = 256
  static constexpr uint32_t IDESC = (1u << 4) | (FMT << 7) | (FMT << 10) |
                                    ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
};

// fused epilogue on 4 consecutive columns (n .. n+3) of row m, all in range, ep.vec_ok
__device__ __forceinline__ void epi4(const Epilogue& ep, float4 t, long long m, int n) {
  float v[4] = {t.x, t.y, t.z, t.w};
  epi_apply4(ep, v, m, n);
}

// ---- staged store of one finished 32-row x W-column piece of the tile ---------------------------------------------
// Lane r owns row r of the piece (the TMEM layout).  It converts its W values into the output plane's format and
// writes them as 16-byte chunks into a [32 rows][RB bytes] staging box (RB = 32, 64 or 128; chunk index XOR-swizzled
// so that neither side has bank conflicts); after a warp sync the box goes out with lanes mapped to (row, chunk), so
// every store instruction writes whole RB-byte row segments.
template <int RB>
__device__ __forceinline__ uint32_t stage_off(int row, int chunk) {
  constexpr int CPR = RB / 16, RPL = 128 / RB;
  return (uint32_t)(row * RB + (((chunk ^ ((row / RPL) % CPR))) << 4));
}
// explicit shared-space accesses on 32-bit addresses: a generic pointer into dynamic shared memory makes the compiler
// re-derive the shared window (S2UR SR_CgaCtaId + address arithmetic) at every access inside a cluster kernel
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void stg128(void* p, uint4 v) {
  asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// four fp32 values added to memory (split-K partial tiles): one vector reduction per 16 bytes
__device__ __forceinline__ void red_add128(void* p, uint4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)),
               "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w)) : "memory");
}
template <int RB>
__device__ __forceinline__ void stage_copy_out(uint32_t stage, int lane, uint8_t* plane, long long ld_bytes,
                                               long long row0, long long M, int col_bytes0, int n_bytes, bool atomic = false) {
  // plane + row * ld_bytes + col_bytes0 is the first byte of the box in global memory; n_bytes = row length in bytes
  constexpr int CPR = RB / 16, ROWS_PER_IT = 32 / CPR;
  const int chunk = lane % CPR, rsub = lane / CPR;
  if (col_bytes0 + chunk * 16 >= n_bytes) return;
  uint8_t* g = plane + (row0 + rsub) * ld_bytes + col_bytes0 + chunk * 16;
  uint4 t[CPR];
#pragma unroll
  for (int it = 0; it < CPR; ++it) t[it] = lds128(stage + stage_off<RB>(it * ROWS_PER_IT + rsub, chunk));
#pragma unroll
  for (int it = 0; it < CPR; ++it)
    if (row0 + it * ROWS_PER_IT + rsub < M) {
      if (atomic) red_add128(g + (long long)it * ROWS_PER_IT * ld_bytes, t[it]);
      else stg128(g + (long long)it * ROWS_PER_IT * ld_bytes, t[it]);
    }
}

// The epilogue description, read ONCE per thread into registers.  Reading the fields from the kernel-parameter
// constant bank where they are used costs a dependent constant load + compare + branch per feature and per group of
// columns (~10^3 cycles per 32-column piece, measured with an in-kernel cycle-counter timeline) -- the pieces must run on registers.
struct EpiRegs {
  uint32_t flags;
  float sign;
  const float* bias;
  const __half* rh;
  const __half* rl;
  __half* oh;
  __half* ol;
  float* of32;
  int ldr16, ld16, ldf32;    // row pitches in elements
};
constexpr uint32_t EF_BIAS = 1, EF_RELU = 2, EF_RESID16 = 4, EF_OUT16 = 8, EF_OUTF32 = 16, EF_RARE = 32, EF_RESID32 = 64,
                   EF_OUTSPLIT = 128, EF_OUTBF16 = 256, EF_ATOMIC = 512;

template <class T>
__device__ __forceinline__ T* launder_ptr(T* p) {   // opaque to the compiler: stays in a register pair
  unsigned long long u = reinterpret_cast<unsigned long long>(p);
  asm volatile("" : "+l"(u));
  return reinterpret_cast<T*>(u);
}
__device__ __forceinline__ EpiRegs load_epi_regs(const Epilogue& ep) {
  EpiRegs r;
  uint32_t f = 0;
  if (ep.bias) f |= EF_BIAS;
  if (ep.relu) f |= EF_RELU;
  if (ep.resid_h16) f |= EF_RESID16;
  if (ep.out_h16) f |= EF_OUT16;
  if (ep.out_f32) f |= EF_OUTF32;
  if (ep.resid_hi) f |= EF_RESID32;
  if (ep.out_hi) f |= EF_OUTSPLIT;
  if (ep.out_bf16) f |= EF_OUTBF16;
  if (ep.colscale || ep.postsub) f |= EF_RARE;
  if (ep.atomic_out) f |= EF_ATOMIC;
  asm volatile("" : "+r"(f));
  r.flags = f;
  r.sign = ep.resid_sign;
  asm volatile("" : "+f"(r.sign));
  r.bias = launder_ptr(ep.bias);
  r.rh = launder_ptr(ep.resid_h16);
  r.rl = launder_ptr(ep.resid_l16);
  r.oh = launder_ptr(ep.out_h16);
  r.ol = launder_ptr(ep.out_l16);
  r.of32 = launder_ptr(ep.out_f32);
  r.ldr16 = (int)ep.ldr_16;
  r.ld16 = (int)ep.ld_16;
  r.ldf32 = (int)ep.ld_f32;
  asm volatile("" : "+r"(r.ldr16), "+r"(r.ld16), "+r"(r.ldf32));
  return r;
}

template <int W>
__device__ __forceinline__ void store_chunk(const Epilogue& ep, const EpiRegs& er, float (&v)[W], long long row0, int lane,
                                            long long M, int n0, int N, uint32_t stage, int path_flags) {
  const long long m = row0 + lane;
  const uint32_t f = er.flags;
  if (m < M) {
    if (f & EF_RARE) {        // column scale / post-subtract / fp32 residual planes: the generic arithmetic
#pragma unroll
      for (int i = 0; i < W; i += 4) {
        if (n0 + i < N) {     // N % 8 == 0 on this path: a group of four is inside or outside as a whole
          float t[4] = {v[i], v[i + 1], v[i + 2], v[i + 3]};
          epi_math4(ep, t, m, n0 + i);
          v[i] = t[0]; v[i + 1] = t[1]; v[i + 2] = t[2]; v[i + 3] = t[3];
        }
      }
    } else {
      if (f & EF_BIAS) {
        const float4* pb = reinterpret_cast<const float4*>(er.bias + n0);
#pragma unroll
        for (int q = 0; q < W / 8; ++q) {
          if (n0 + q * 8 < N) {
            const float4 b0 = __ldg(pb + 2 * q), b1 = __ldg(pb + 2 * q + 1);
            v[8 * q] += b0.x; v[8 * q + 1] += b0.y; v[8 * q + 2] += b0.z; v[8 * q + 3] += b0.w;
            v[8 * q + 4] += b1.x; v[8 * q + 5] += b1.y; v[8 * q + 6] += b1.z; v[8 * q + 7] += b1.w;
          }
        }
      }
      if (f & EF_RELU) {
#pragma unroll
        for (int i = 0; i < W; ++i) v[i] = fmaxf(v[i], 0.f);
      }
      if (f & EF_RESID16) {   // coupling: x -/+ t with x in fp16 split planes
        const uint4* ph = reinterpret_cast<const uint4*>(er.rh + m * er.ldr16 + n0);
        const uint4* pl = reinterpret_cast<const uint4*>(er.rl + m * er.ldr16 + n0);
#pragma unroll
        for (int q = 0; q < W / 8; ++q) {
          if (n0 + q * 8 < N) {
            const uint4 h8 = ph[q], l8 = pl[q];
            const __half2* h2 = reinterpret_cast<const __half2*>(&h8);
            const __half2* l2 = reinterpret_cast<const __half2*>(&l8);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 hf = __half22float2(h2[e]), lf = __half22float2(l2[e]);
              v[8 * q + 2 * e] = fmaf(er.sign, v[8 * q + 2 * e], fmaf(lf.x, F16_LO_UNSCALE, hf.x));
              v[8 * q + 2 * e + 1] = fmaf(er.sign, v[8 * q + 2 * e + 1], fmaf(lf.y, F16_LO_UNSCALE, hf.y));
            }
          }
        }
      }
      if (f & EF_RESID32) {   // fp32 residual stream (bf16 mode) or tf32 split planes (hi + lo)
        // (the engines other than the fp16-split one: their pointers are read from the parameter bank once per piece)
        const float* r32lo = ep.resid_lo;
        const float4* pr = reinterpret_cast<const float4*>(ep.resid_hi + m * ep.ldr + n0);
        const float4* pl = reinterpret_cast<const float4*>(r32lo + m * ep.ldr + n0);
#pragma unroll
        for (int q = 0; q < W / 4; ++q) {
          if (n0 + q * 4 < N) {
            float4 r = pr[q];
            if (r32lo) {
              const float4 l = pl[q];
              r.x += l.x; r.y += l.y; r.z += l.z; r.w += l.w;
            }
            v[4 * q] = fmaf(er.sign, v[4 * q], r.x); v[4 * q + 1] = fmaf(er.sign, v[4 * q + 1], r.y);
            v[4 * q + 2] = fmaf(er.sign, v[4 * q + 2], r.z); v[4 * q + 3] = fmaf(er.sign, v[4 * q + 3], r.w);
          }
        }
      }
    }
  }
  if (f & EF_OUT16) {      // fp16 split planes: x = hi + lo' 2^-11
    constexpr int RB = W * 2;
    const uint32_t stage_lo = stage + 32 * RB;
    // debug flag 16: register-direct stores.  Unused, but deleting it shifts ptxas' register allocation and slowed the
    // BLOCK_N = 256 3xTF32 instantiation by 2% (1024 x 1024 over 65 536 rows, B200)
    const bool direct = (path_flags & 16) != 0;
    uint4* gh = reinterpret_cast<uint4*>(er.oh + m * er.ld16 + n0);
    uint4* gl = reinterpret_cast<uint4*>(er.ol + m * er.ld16 + n0);
    __half2 amax2 = __float2half2_rn(0.f);      // running max |hi| (NaN-propagating): inf / NaN = the value left the fp16 range
#pragma unroll
    for (int q = 0; q < W / 8; ++q) {
      uint32_t hp[4], lp[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float x0 = v[q * 8 + 2 * e], x1 = v[q * 8 + 2 * e + 1];
        const __half2 h = __floats2half2_rn(x0, x1);
        const float2 hf = __half22float2(h);
        const __half2 l = __floats2half2_rn((x0 - hf.x) * F16_LO_SCALE, (x1 - hf.y) * F16_LO_SCALE);
        hp[e] = *reinterpret_cast<const uint32_t*>(&h);
        lp[e] = *reinterpret_cast<const uint32_t*>(&l);
        if (n0 + q * 8 < N) amax2 = __hmax2_nan(amax2, __habs2(h));
      }
      if (direct) {
        if (m < M && n0 + q * 8 < N) {
          gh[q] = make_uint4(hp[0], hp[1], hp[2], hp[3]);
          gl[q] = make_uint4(lp[0], lp[1], lp[2], lp[3]);
        }
      } else {
        sts128(stage + stage_off<RB>(lane, q), hp[0], hp[1], hp[2], hp[3]);
        sts128(stage_lo + stage_off<RB>(lane, q), lp[0], lp[1], lp[2], lp[3]);
      }
    }
    {
      const float2 am = __half22float2(amax2);
      if (!(am.x <= F16_GUARD && am.y <= F16_GUARD) && m < M && ep.overflow_flag) *ep.overflow_flag = 1;
    }
    if (!direct) {
      __syncwarp();
      stage_copy_out<RB>(stage, lane, reinterpret_cast<uint8_t*>(er.oh), (long long)er.ld16 * 2, row0, M, n0 * 2, N * 2);
      stage_copy_out<RB>(stage_lo, lane, reinterpret_cast<uint8_t*>(er.ol), (long long)er.ld16 * 2, row0, M, n0 * 2, N * 2);
      __syncwarp();
    }
  }
  if (f & EF_OUTF32) {
    constexpr int RB = W * 4;
#pragma unroll
    for (int q = 0; q < W / 4; ++q)
      sts128(stage + stage_off<RB>(lane, q), __float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]), __float_as_uint(v[4 * q + 2]),
             __float_as_uint(v[4 * q + 3]));
    __syncwarp();
    stage_copy_out<RB>(stage, lane, reinterpret_cast<uint8_t*>(er.of32), (long long)er.ldf32 * 4, row0, M, n0 * 4, N * 4,
                       (f & EF_ATOMIC) != 0);
    __syncwarp();
  }
  {
    if (f & EF_OUTBF16) {
      constexpr int RB = W * 2;
#pragma unroll
      for (int q = 0; q < W / 8; ++q) {
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const __nv_bfloat162 t = __floats2bfloat162_rn(v[q * 8 + 2 * e], v[q * 8 + 2 * e + 1]);
          pk[e] = *reinterpret_cast<const uint32_t*>(&t);
        }
        sts128(stage + stage_off<RB>(lane, q), pk[0], pk[1], pk[2], pk[3]);
      }
      __syncwarp();
      stage_copy_out<RB>(stage, lane, reinterpret_cast<uint8_t*>(ep.out_bf16), ep.ld_bf16 * 2, row0, M, n0 * 2, N * 2);
      __syncwarp();
    }
    if (f & EF_OUTSPLIT) {   // tf32 split planes
      constexpr int RB = W * 4;
#pragma unroll
      for (int q = 0; q < W / 4; ++q)
        sts128(stage + stage_off<RB>(lane, q), __float_as_uint(tf32_round(v[4 * q])), __float_as_uint(tf32_round(v[4 * q + 1])),
               __float_as_uint(tf32_round(v[4 * q + 2])), __float_as_uint(tf32_round(v[4 * q + 3])));
      __syncwarp();
      stage_copy_out<RB>(stage, lane, reinterpret_cast<uint8_t*>(ep.out_hi), ep.ld_split * 4, row0, M, n0 * 4, N * 4);
      __syncwarp();
#pragma unroll
      for (int q = 0; q < W / 4; ++q)
        sts128(stage + stage_off<RB>(lane, q), __float_as_uint(tf32_round(v[4 * q] - tf32_round(v[4 * q]))),
               __float_as_uint(tf32_round(v[4 * q + 1] - tf32_round(v[4 * q + 1]))),
               __float_as_uint(tf32_round(v[4 * q + 2] - tf32_round(v[4 * q + 2]))),
               __float_as_uint(tf32_round(v[4 * q + 3] - tf32_round(v[4 * q + 3]))));
      __syncwarp();
      stage_copy_out<RB>(stage, lane, reinterpret_cast<uint8_t*>(ep.out_lo), ep.ld_split * 4, row0, M, n0 * 4, N * 4);
      __syncwarp();
    }
  }
}

// ---- asynchronous store path (fp16-split planes only) ---------------------------------------------------------------
// The epilogue warp converts W = 32 columns of its row at a time (16 for the tail of a 112 / 96 column range), FIRST the
// hi plane into staging box A, THEN the lo plane into box B; one lane issues a TMA tensor store per box.  Rows of a box
// are W * 2 = 64 bytes (hardware 64B swizzle; 32B for the tail): whole 64-byte segments per row on the SM -> L2 write
// path, which is what bounds this phase.  Each plane has its own box, so a box is rewritten two store groups later
// (`cp.async.bulk.wait_group.read 1`): the stores run under the conversion of the next plane / piece and under the next
// tile's main loop, and the M / N edges are clipped by the hardware.
struct StoreMaps { CUtensorMap h32, l32, h16, l16; };    // [M rows, N cols] fp16; box = 32 rows x 32 (64B swizzle) / 16 columns (32B)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
constexpr int ASYNC_BOX_BYTES = 32 * 32 * 2;       // one 32-row x 32-column fp16 box = 2 KB (box A at +0, box B at +2 KB)

// Coupling residual, read COALESCED.  A lane owns one row of the piece (the TMEM layout), but 32 lanes reading 16 bytes
// of 32 different rows cost one LSU tag lookup per lane and instruction (measured: +80 us on the 392 x 1024 layer of C2,
// profiles/r01_timeline_pair_f16.md).  Here the warp reads the piece with lanes mapped to (row group, 16-byte chunk) --
// every load instruction covers whole RB-byte row segments of 32 / CPR rows -- drops it into the warp's in-box (same
// XOR swizzle as the staging boxes: conflict-free both ways) and every lane picks its own row up from there.
__device__ __forceinline__ uint4 ldg128(const void* p) {
  uint4 v;
  asm volatile("ld.global.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
template <int W>
__device__ __forceinline__ void coop_resid_row(const __half* plane, int ldr, long long row0, long long M, int n0, int N, int lane,
                                               uint32_t inbox, uint4 (&row)[W / 8]) {
  constexpr int RB = W * 2, CPR = RB / 16, RPI = 32 / CPR;
  const int chunk = lane % CPR, rsub = lane / CPR;
  uint4 t[CPR];
  const bool col_ok = n0 + chunk * 8 < N;
#pragma unroll
  for (int it = 0; it < CPR; ++it) {
    const long long r = row0 + rsub + RPI * it;
    t[it] = make_uint4(0u, 0u, 0u, 0u);
    if (col_ok && r < M) t[it] = ldg128(plane + r * ldr + n0 + chunk * 8);
  }
#pragma unroll
  for (int it = 0; it < CPR; ++it) sts128(inbox + stage_off<RB>(rsub + RPI * it, chunk), t[it].x, t[it].y, t[it].z, t[it].w);
  __syncwarp();
#pragma unroll
  for (int q = 0; q < W / 8; ++q) row[q] = lds128(inbox + stage_off<RB>(lane, q));
  __syncwarp();          // every lane has its row: the box may be rewritten
}

// `bias4` = this lane's four bias values of the warp's column range (lane l holds columns 4l .. 4l+3 of the range,
// loaded once per tile before the last drain); the piece starting at column `c_first` of the range takes its values
// from lanes c_first/4 .. by shuffle, so no global load sits between two TMA stores
template <int W>
__device__ __forceinline__ void async_math(const Epilogue& ep, const EpiRegs& er, float (&v)[W], const float4& bias4, int c_first,
                                           long long m, bool row_ok, int n0, int N, long long row0, long long M, int lane,
                                           uint32_t inbox) {
  const uint32_t f = er.flags;
  if (f & EF_BIAS) {                 // (all lanes take part in the shuffles)
#pragma unroll
    for (int q = 0; q < W / 4; ++q) {
      const int src = c_first / 4 + q;
      v[4 * q] += __shfl_sync(0xffffffffu, bias4.x, src);
      v[4 * q + 1] += __shfl_sync(0xffffffffu, bias4.y, src);
      v[4 * q + 2] += __shfl_sync(0xffffffffu, bias4.z, src);
      v[4 * q + 3] += __shfl_sync(0xffffffffu, bias4.w, src);
    }
  }
  if ((f & EF_RESID16) && inbox != 0) {   // (all lanes take part: rows past M load nothing and use nothing)
    uint4 rowh[W / 8], rowl[W / 8];
    coop_resid_row<W>(er.rh, er.ldr16, row0, M, n0, N, lane, inbox, rowh);
    coop_resid_row<W>(er.rl, er.ldr16, row0, M, n0, N, lane, inbox, rowl);
    if (!row_ok) return;
    if (f & EF_RELU) {
#pragma unroll
      for (int i = 0; i < W; ++i) v[i] = fmaxf(v[i], 0.f);
    }
#pragma unroll
    for (int q = 0; q < W / 8; ++q) {
      if (n0 + 8 * q < N) {
        const __half2* h2 = reinterpret_cast<const __half2*>(&rowh[q]);
        const __half2* l2 = reinterpret_cast<const __half2*>(&rowl[q]);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 hf = __half22float2(h2[e]), lf = __half22float2(l2[e]);
          v[8 * q + 2 * e] = fmaf(er.sign, v[8 * q + 2 * e], fmaf(lf.x, F16_LO_UNSCALE, hf.x));
          v[8 * q + 2 * e + 1] = fmaf(er.sign, v[8 * q + 2 * e + 1], fmaf(lf.y, F16_LO_UNSCALE, hf.y));
        }
      }
    }
    return;
  }
  if (!row_ok) return;
  if (f & EF_RELU) {
#pragma unroll
    for (int i = 0; i < W; ++i) v[i] = fmaxf(v[i], 0.f);
  }
  if (f & EF_RESID16) {   // coupling: x -/+ t with x in fp16 split planes (possibly the planes being written: in place)
    const uint4* ph = reinterpret_cast<const uint4*>(er.rh + m * er.ldr16 + n0);
    const uint4* pl = reinterpret_cast<const uint4*>(er.rl + m * er.ldr16 + n0);
#pragma unroll
    for (int q = 0; q < W / 8; ++q) {
      if (n0 + 8 * q < N) {          // N % 8 == 0: a group of eight columns is inside or outside as a whole
        const uint4 h8 = ph[q], l8 = pl[q];
        const __half2* h2 = reinterpret_cast<const __half2*>(&h8);
        const __half2* l2 = reinterpret_cast<const __half2*>(&l8);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 hf = __half22float2(h2[e]), lf = __half22float2(l2[e]);
          v[8 * q + 2 * e] = fmaf(er.sign, v[8 * q + 2 * e], fmaf(lf.x, F16_LO_UNSCALE, hf.x));
          v[8 * q + 2 * e + 1] = fmaf(er.sign, v[8 * q + 2 * e + 1], fmaf(lf.y, F16_LO_UNSCALE, hf.y));
        }
      }
    }
  }
  if (f & EF_RESID32) {   // fp32 residual stream (bf16 / tf32 modes); same arithmetic as store_chunk
    const float* r32lo = ep.resid_lo;
    const float4* pr = reinterpret_cast<const float4*>(ep.resid_hi + m * ep.ldr + n0);
    const float4* pl = reinterpret_cast<const float4*>(r32lo + m * ep.ldr + n0);
#pragma unroll
    for (int q = 0; q < W / 4; ++q) {
      if (n0 + q * 4 < N) {
        float4 r = pr[q];
        if (r32lo) {
          const float4 l = pl[q];
          r.x += l.x; r.y += l.y; r.z += l.z; r.w += l.w;
        }
        v[4 * q] = fmaf(er.sign, v[4 * q], r.x); v[4 * q + 1] = fmaf(er.sign, v[4 * q + 1], r.y);
        v[4 * q + 2] = fmaf(er.sign, v[4 * q + 2], r.z); v[4 * q + 3] = fmaf(er.sign, v[4 * q + 3], r.w);
      }
    }
  }
}

// one plane (LO = false: hi, true: lo' = (x - hi) 2^11) of a W-column piece -> staging box (row = lane)
template <int W, bool LO>
__device__ __forceinline__ void async_stage_plane(const Epilogue& ep, const float (&v)[W], bool row_ok, int lane, int n0, int N,
                                                  uint32_t box) {
  constexpr int RB = W * 2;
  __half2 amax2 = __float2half2_rn(0.f);
#pragma unroll
  for (int q = 0; q < W / 8; ++q) {
    uint32_t pk[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x0 = v[q * 8 + 2 * e], x1 = v[q * 8 + 2 * e + 1];
      const __half2 h = __floats2half2_rn(x0, x1);
      if (LO) {
        const float2 hf = __half22float2(h);
        const __half2 l = __floats2half2_rn((x0 - hf.x) * F16_LO_SCALE, (x1 - hf.y) * F16_LO_SCALE);
        pk[e] = *reinterpret_cast<const uint32_t*>(&l);
      } else {
        pk[e] = *reinterpret_cast<const uint32_t*>(&h);
        if (n0 + 8 * q < N) amax2 = __hmax2_nan(amax2, __habs2(h));   // columns past N hold no result
      }
    }
    sts128(box + stage_off<RB>(lane, q), pk[0], pk[1], pk[2], pk[3]);
  }
  if (!LO) {
    const float2 am = __half22float2(amax2);
    if (!(am.x <= F16_GUARD && am.y <= F16_GUARD) && row_ok && ep.overflow_flag) *ep.overflow_flag = 1;
  }
}

// a whole W-column piece: arithmetic, then plane by plane: wait for the box, stage, TMA store
template <int W>
__device__ __forceinline__ void async_piece(const Epilogue& ep, const EpiRegs& er, const StoreMaps& smaps, float (&v)[W],
                                            const float4& bias4, int c_first, long long m, bool row_ok, int lane, int n0, int N,
                                            long long row0, uint32_t stage, uint32_t& groups, long long M, uint32_t inbox) {
  async_math<W>(ep, er, v, bias4, c_first, m, row_ok, n0, N, row0, M, lane, inbox);
  const CUtensorMap* mh = W == 32 ? &smaps.h32 : &smaps.h16;
  const CUtensorMap* ml = W == 32 ? &smaps.l32 : &smaps.l16;
#pragma unroll
  for (int plane = 0; plane < 2; ++plane) {
    if (groups >= 2) {                                // the store that last read this box (two groups ago) has drained it
      if (lane == 0) bulk_wait_read1();
      __syncwarp();
    }
    const uint32_t box = stage + plane * ASYNC_BOX_BYTES;
    if (plane == 0) async_stage_plane<W, false>(ep, v, row_ok, lane, n0, N, box);
    else async_stage_plane<W, true>(ep, v, row_ok, lane, n0, N, box);
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(plane == 0 ? mh : ml, box, n0, (int)row0);
      bulk_commit();
    }
    ++groups;
  }
}

// Mode 2 of the asynchronous store path: a bf16 plane and / or an fp32 plane (bf16 and tf32 precision modes).  Same two
// 2 KB boxes per warp, used in turn: the bf16 piece is 32 rows x 32 columns (64-byte rows, map h32; 16 columns / 32-byte rows
// for the tail, map h16), the fp32 piece goes out as 16-column halves (64-byte rows, map l32).  In these modes the store
// phase was the largest part of a launch (1024 x 1024 over 65 536 rows, bf16: 153.8 us, 102.9 us with the store phase off).
template <int W>
__device__ __forceinline__ void async_piece2(const Epilogue& ep, const EpiRegs& er, const StoreMaps& smaps, float (&v)[W],
                                             const float4& bias4, int c_first, long long m, bool row_ok, int lane, int n0, int N,
                                             long long row0, uint32_t stage, uint32_t& groups, long long M) {
  async_math<W>(ep, er, v, bias4, c_first, m, row_ok, n0, N, row0, M, lane, 0u);
  if (er.flags & EF_OUTBF16) {
    constexpr int RB = W * 2;
    if (groups >= 2) {
      if (lane == 0) bulk_wait_read1();
      __syncwarp();
    }
    const uint32_t box = stage + (groups & 1u) * ASYNC_BOX_BYTES;
#pragma unroll
    for (int q = 0; q < W / 8; ++q) {
      uint32_t pk[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const __nv_bfloat162 t = __floats2bfloat162_rn(v[q * 8 + 2 * e], v[q * 8 + 2 * e + 1]);
        pk[e] = *reinterpret_cast<const uint32_t*>(&t);
      }
      sts128(box + stage_off<RB>(lane, q), pk[0], pk[1], pk[2], pk[3]);
    }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(W == 32 ? &smaps.h32 : &smaps.h16, box, n0, (int)row0);
      bulk_commit();
    }
    ++groups;
  }
  if (er.flags & EF_OUTF32) {
#pragma unroll
    for (int half = 0; half < W / 16; ++half) {
      if (n0 + 16 * half < N) {
        if (groups >= 2) {
          if (lane == 0) bulk_wait_read1();
          __syncwarp();
        }
        const uint32_t box = stage + (groups & 1u) * ASYNC_BOX_BYTES;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          sts128(box + stage_off<64>(lane, q), __float_as_uint(v[16 * half + 4 * q]), __float_as_uint(v[16 * half + 4 * q + 1]),
                 __float_as_uint(v[16 * half + 4 * q + 2]), __float_as_uint(v[16 * half + 4 * q + 3]));
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&smaps.l32, box, n0 + 16 * half, (int)row0);
          bulk_commit();
        }
        ++groups;
      }
    }
  }
}

// One epilogue warp: TMEM lanes [32*quarter, +32) x columns [col0, col0+COLS) of every tile of this CTA.
template <class C, int COLS, bool SPLITK>
__device__ __forceinline__ void epilogue_loop(int col0, int quarter, int lane, uint32_t rank, uint32_t tmem_base,
                                              uint32_t tfull0, uint32_t tempty0_leader, uint8_t* stage_gen,
                                              uint32_t stage, long long n_tiles, int n_blocks, int k_slabs, int split_k, int split_per, int chunk_slabs, int lead,
                                              long long M, int N, const Epilogue& ep, int path_flags, const StoreMaps& smaps) {
  constexpr int BLOCK_N = C::kBlockN;
  int acc = 0;
  uint32_t acc_phase = 0;
  int n_chunks = chain_count(k_slabs, chunk_slabs, lead);   // (split_k == 1; recomputed per work item otherwise)
  float* patch = reinterpret_cast<float*>(stage_gen);
  // everything the tile loop needs lives in registers from here on (opaque to the compiler): re-deriving these from
  // special registers / the parameter bank inside the loop costs a dependent S2R / LDC per use
  asm volatile("" : "+r"(stage), "+r"(tfull0), "+r"(tempty0_leader), "+r"(tmem_base));
  // the warp's in-box sits right behind its staging boxes (no register of its own); path flag 256 switches it off
  const uint32_t inbox = (C::INBOX && !(path_flags & 256)) ? stage + STAGE_EPI_BYTES : 0u;
  asm volatile("" : "+l"(M), "+r"(N), "+r"(lane), "+r"(quarter), "+r"(col0), "+r"(rank), "+r"(n_blocks), "+l"(n_tiles),
               "+r"(n_chunks), "+r"(path_flags));
  const EpiRegs er = load_epi_regs(ep);
  const bool fast_store = ep.fast_store != 0;
  const bool async_store = ep.async_store != 0;
  const bool async_wide = ep.async_store == 2;      // bf16 / fp32 planes (async_piece2)
  uint32_t hand = 0;     // TMA store groups committed so far by this warp
  for (long long tile = cluster_id_x(); tile < n_tiles; tile += num_clusters_x()) {
    long long m_blk = tile / n_blocks;
    int n_blk = (int)(tile % n_blocks);
    if (SPLITK) {
      const TileCoord tc = decode_tile<true>(tile, n_blocks, split_k, k_slabs, split_per);
      m_blk = tc.m_blk;
      n_blk = tc.n_blk;
      n_chunks = chain_count(tc.nks, chunk_slabs, lead);
    }
    const long long m_idx = m_blk * (2 * BLOCK_M) + rank * BLOCK_M;
    const int n_idx = n_blk * BLOCK_N;
    if (COLS == 0) {  // nothing to own: still take part in the barrier protocol
      for (int c = 0; c < n_chunks; ++c) {
        mbar_wait(tfull0 + 8u * acc, acc_phase);
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty0_leader + 8u * acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      continue;
    }
    // partial accumulators (one per K chunk) are added in place with round-to-nearest; starting from zero keeps
    // one register copy of the tile (a "first chunk moves, later chunks add" split doubles the live registers)
    float master[COLS > 0 ? COLS : 1];
#pragma unroll
    for (int i = 0; i < COLS; ++i) master[i] = 0.f;
    float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < n_chunks; ++c) {
      if (c == n_chunks - 1 && async_store && (er.flags & EF_BIAS)) {   // in flight during the last drain
        const int nb = n_idx + col0 + 4 * lane;
        if (4 * lane < COLS && nb < N) bias4 = __ldg(reinterpret_cast<const float4*>(er.bias + nb));
      }
      mbar_wait(tfull0 + 8u * acc, acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * C::ACC_STRIDE + col0;
#pragma unroll
      for (int j = 0; j + 32 <= COLS; j += 32) {
        if (n_idx + col0 + j < N) {      // columns past N hold no MMA result (the last tile of a row may be narrower)
          float v[32];
          tmem_ld32(taddr + j, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) master[j + i] += v[i];
        }
      }
      if (COLS % 32) {
        constexpr int j = COLS / 32 * 32;
        if (n_idx + col0 + j < N) {
          float v[16];
          tmem_ld16(taddr + j, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) master[j + i] += v[i];
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty0_leader + 8u * acc);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    const long long row0 = m_idx + quarter * 32;
    if (async_store) {
      if (row0 < M) {
        const long long m = row0 + lane;
        const bool row_ok = m < M;
#pragma unroll
        for (int c = 0; c < COLS / 32; ++c) {
          const int n0 = n_idx + col0 + c * 32;
          if (n0 < N) {
            if (async_wide)
              async_piece2<32>(ep, er, smaps, *reinterpret_cast<float(*)[32]>(&master[c * 32]), bias4, c * 32, m, row_ok, lane,
                               n0, N, row0, stage, hand, M);
            else
              async_piece<32>(ep, er, smaps, *reinterpret_cast<float(*)[32]>(&master[c * 32]), bias4, c * 32, m, row_ok, lane,
                              n0, N, row0, stage, hand, M, inbox);
          }
        }
        if (COLS % 32) {
          constexpr int c_first = COLS / 32 * 32;
          const int n0 = n_idx + col0 + c_first;
          if (n0 < N) {
            if (async_wide)
              async_piece2<16>(ep, er, smaps, *reinterpret_cast<float(*)[16]>(&master[c_first]), bias4, c_first, m, row_ok, lane,
                               n0, N, row0, stage, hand, M);
            else
              async_piece<16>(ep, er, smaps, *reinterpret_cast<float(*)[16]>(&master[c_first]), bias4, c_first, m, row_ok, lane,
                              n0, N, row0, stage, hand, M, inbox);
          }
        }
      }
    } else if (fast_store) {
      if (row0 < M) {
#pragma unroll
        for (int c = 0; c < COLS / 32; ++c) {
          const int n0 = n_idx + col0 + c * 32;
          if (n0 < N)
            store_chunk<32>(ep, er, *reinterpret_cast<float(*)[32]>(&master[c * 32]), row0, lane, M, n0, N, stage, path_flags);
        }
        if (COLS % 32) {
          const int n0 = n_idx + col0 + COLS / 32 * 32;
          if (n0 < N) store_chunk<16>(ep, er, *reinterpret_cast<float(*)[16]>(&master[COLS / 32 * 32]), row0, lane, M, n0, N, stage, path_flags);
        }
      }
    } else {
      // unaligned output planes: registers -> padded smem patch -> 64 B row segments (4 lanes x 16 B per row)
      const int sub_r = lane >> 2, sub_c = (lane & 3) * 4;
#pragma unroll
      for (int j = 0; j < COLS; j += PATCH_COLS) {
        float* prow = patch + lane * PATCH_LD;
#pragma unroll
        for (int i = 0; i < PATCH_COLS; i += 4)
          *reinterpret_cast<float4*>(prow + i) = make_float4(master[j + i], master[j + i + 1], master[j + i + 2], master[j + i + 3]);
        __syncwarp();
        const int n = n_idx + col0 + j + sub_c;
#pragma unroll 1
        for (int p = 0; p < 4; ++p) {
          const int r = p * 8 + sub_r;
          const long long m = row0 + r;
          const float4 t = *reinterpret_cast<const float4*>(patch + r * PATCH_LD + sub_c);
          if (m < M && n < N) {
            if (ep.vec_ok && n + 3 < N) {
              epi4(ep, t, m, n);
            } else {
              const float tv[4] = {t.x, t.y, t.z, t.w};
              for (int i = 0; i < 4; ++i)
                if (n + i < N) epi_store1(ep, epi_value(ep, tv[i], m, n + i), m, n + i);
            }
          }
        }
        __syncwarp();
      }
    }
  }
  if (async_store && lane == 0) bulk_wait0();   // staging memory and the stores outlive their reads / writes
  __syncwarp();
}

template <int BLOCK_N, int NTERMS, int KIND, bool SPLITK = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_a_lo,
                const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_w_lo,
                long long M, int N, int K, int chunk_slabs, int lead_chains, int split_k, int split_per,
                const __grid_constant__ Epilogue ep, const __grid_constant__ StoreMaps smaps, int path_flags) {
  using C = Config<BLOCK_N, NTERMS, KIND>;
  extern __shared__ uint8_t smem_raw[];
  uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // same offset in both CTAs of the pair
  asm volatile("" : "+r"(smem_base));   // opaque: otherwise every use re-derives it (S2UR SR_CgaCtaId + arithmetic)
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t epi_base = smem_base + C::STAGES * C::STAGE_BYTES;
  const uint32_t bar_base = epi_base + C::EPI_BYTES;
  // barrier block: full[STAGES] (leader's is used), empty[STAGES], tmem_full[2], tmem_empty[2] (leader's), tmem slot
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (C::STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * C::STAGES + 4);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int n_blocks = (N + BLOCK_N - 1) / BLOCK_N;
  const long long m_blocks = (M + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
  const int k_slabs = (K + C::ELEMS_PER_SLAB - 1) / C::ELEMS_PER_SLAB;
  if (!SPLITK || split_k < 1) split_k = 1;
  const long long n_tiles = m_blocks * n_blocks * split_k;
  if (chunk_slabs <= 0 || chunk_slabs > k_slabs) chunk_slabs = k_slabs;
  if (KIND == KIND_F16 && NTERMS == 3) chunk_slabs = 1;   // one K-slab = 64 K-elements per accumulation chain (the 2^-11
                                                         // rescale happens once per chain)
  // the last tile of a tile row is only as wide as N needs (UMMA N is a run-time field of the instruction descriptor;
  // multiples of 16 for M = 256), and the last K-slab only issues the 32-byte K steps that hold data
  auto tile_width = [&](int n_idx) {
    const int rest = (N - n_idx + 15) & ~15;
    return rest < 32 ? 32 : rest < BLOCK_N ? rest : BLOCK_N;
  };
  const int last_ksteps = ((K - (k_slabs - 1) * C::ELEMS_PER_SLAB) * (SLAB_BYTES / C::ELEMS_PER_SLAB) + UMMA_K_BYTES - 1) / UMMA_K_BYTES;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a);
    prefetch_tmap(&tm_w);
    if (NTERMS == 3) { prefetch_tmap(&tm_a_lo); prefetch_tmap(&tm_w_lo); }
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
      for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 2 * NUM_EPI_WARPS); }
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();      // (orders the allocator's write of the TMEM base address for this CTA's readers: a plain CTA barrier,
                        //  which compute-sanitizer's racecheck tracks -- it does not model barrier.cluster)
  cluster_sync_all();   // barriers of both CTAs initialised and visible before any remote arrive / TMA completion
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // everything above touched only this CTA's shared / tensor memory and kernel parameters: it may run while the previous
  // kernel of the chain still drains; from here on global memory written by that kernel is read
  griddep_launch_dependents();
  griddep_wait();

  if (warp < FIRST_EPI_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_NON_EPI));
    if (warp == 0) {
      // ===================== TMA producer (both CTAs) =====================
      // (the issuing thread of each role is picked with elect.sync: the compiler then emits TMA / tcgen05.mma back to back
      //  instead of wrapping each one in an ELECT / BRA.U.ANY loop that waits on the instruction's scoreboard; and ONE
      //  thread runs the barrier protocol -- 32 lanes polling an mbarrier serialise; see csrc/conv_pix.cuh)
      if (elect_one()) {
        int stage = 0;
        uint32_t phase = 0;
        for (long long tile = cluster_id_x(); tile < n_tiles; tile += num_clusters_x()) {
          const TileCoord tc = decode_tile<SPLITK>(tile, n_blocks, split_k, k_slabs, split_per);
          const int m_idx = (int)tc.m_blk * (2 * BLOCK_M) + (int)rank * BLOCK_M;
          const int n_tile = tc.n_blk * BLOCK_N;
          const int n_idx = n_tile + (int)rank * (tile_width(n_tile) >> 1);   // this CTA stages its half of the W rows
          for (int ks = 0; ks < tc.nks; ++ks) {
            mbar_wait(empty_bar(stage), phase ^ 1);
            const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
            const uint32_t sb = sa + C::NPLANES * C::A_TILE;
            const int k_idx = (tc.ks_begin + ks) * C::ELEMS_PER_SLAB;
            const uint32_t fb = mapa(full_bar(stage), 0);
            if (rank == 0) mbar_expect_tx(full_bar(stage), 2 * C::STAGE_BYTES);
            tma_load_2d_pair(sa, &tm_a, fb, k_idx, m_idx);
            tma_load_2d_pair(sb, &tm_w, fb, k_idx, n_idx);
            if (NTERMS == 3) {
              tma_load_2d_pair(sa + C::A_TILE, &tm_a_lo, fb, k_idx, m_idx);
              tma_load_2d_pair(sb + C::B_TILE, &tm_w_lo, fb, k_idx, n_idx);
            }
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    } else if (warp == 1 && rank == 0 && elect_one()) {
      // ===================== MMA issuer (leader CTA only) =====================
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (long long tile = cluster_id_x(); tile < n_tiles; tile += num_clusters_x()) {
        const TileCoord tc = decode_tile<SPLITK>(tile, n_blocks, split_k, k_slabs, split_per);
        const uint32_t idesc = C::IDESC_NO_N | ((uint32_t)(tile_width(tc.n_blk * BLOCK_N) >> 3) << 17);
        const int lead = chain_lead(tc.nks, chunk_slabs, lead_chains);
        const int ks_last = k_slabs - 1 - tc.ks_begin;   // index (within this work item) of the K tail slab, if it is here
        int ks0 = 0;
        for (int c = 0; ks0 < tc.nks; ++c) {
          const int span = c < lead ? 2 * chunk_slabs : chunk_slabs;
          const int ks1 = ks0 + span < tc.nks ? ks0 + span : tc.nks;
          mbar_wait(tempty_bar(acc), acc_phase ^ 1);  // both CTAs' epilogues have drained this accumulator
          tcgen05_fence_after();
          const uint32_t tmem_d = tmem_base + acc * C::ACC_STRIDE;
          constexpr int KSTEPS = SLAB_BYTES / UMMA_K_BYTES;
          if (NTERMS == 3 && KIND == KIND_F16) {
            // fp16 split: the cross terms of EVERY slab of the chain first (their low planes are stored scaled by
            // 2^11), then the first hi.hi product rescales the accumulator by 2^-11, then the other hi.hi products.
            // A chain holds its (1 or 2) pipeline stages until its last product has been issued.
            int st = stage;
            uint32_t ph = phase;
            for (int ks = ks0; ks < ks1; ++ks) {
              mbar_wait(full_bar(st), ph);
              tcgen05_fence_after();
              {
                const uint32_t sa = smem_base + st * C::STAGE_BYTES;
                const uint32_t sb = sa + C::NPLANES * C::A_TILE;
                const uint64_t da_hi = make_smem_desc(sa), db_hi = make_smem_desc(sb);
                const uint64_t da_lo = make_smem_desc(sa + C::A_TILE), db_lo = make_smem_desc(sb + C::B_TILE);
                const int nk = ks == ks_last ? last_ksteps : KSTEPS;
#pragma unroll
                for (int k = 0; k < KSTEPS; ++k) {
                  if (k < nk) {
                    const uint64_t koff = (uint64_t)((k * UMMA_K_BYTES) >> 4);
                    umma_pair<KIND>(da_lo + koff, db_hi + koff, tmem_d, idesc, (ks > ks0 || k > 0) ? 1u : 0u);
                    umma_pair<KIND>(da_hi + koff, db_lo + koff, tmem_d, idesc, 1u);
                  }
                }
              }
              if (++st == C::STAGES) { st = 0; ph ^= 1; }
            }
            for (int ks = ks0; ks < ks1; ++ks) {
              {
                const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
                const uint32_t sb = sa + C::NPLANES * C::A_TILE;
                const uint64_t da_hi = make_smem_desc(sa), db_hi = make_smem_desc(sb);
                const int nk = ks == ks_last ? last_ksteps : KSTEPS;
                if (ks == ks0) umma_pair_f16_scale11(da_hi, db_hi, tmem_d, idesc);
#pragma unroll
                for (int k = 0; k < KSTEPS; ++k) {
                  if (k < nk && (k > 0 || ks > ks0)) {
                    const uint64_t koff = (uint64_t)((k * UMMA_K_BYTES) >> 4);
                    umma_pair<KIND>(da_hi + koff, db_hi + koff, tmem_d, idesc, 1u);
                  }
                }
                umma_commit_pair(empty_bar(stage));                  // slot free in both CTAs once these MMAs retire
                if (ks == ks1 - 1) umma_commit_pair(tfull_bar(acc));  // accumulation chain complete (both CTAs)
              }
              if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            }
          } else {
            for (int ks = ks0; ks < ks1; ++ks) {
              mbar_wait(full_bar(stage), phase);
              tcgen05_fence_after();
              {
                const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
                const uint32_t sb = sa + C::NPLANES * C::A_TILE;
                const uint64_t da_hi = make_smem_desc(sa), db_hi = make_smem_desc(sb);
                const int nk = ks == ks_last ? last_ksteps : KSTEPS;
                if (NTERMS == 3) {  // small terms first: they meet the accumulator while it is smallest
                  const uint64_t da_lo = make_smem_desc(sa + C::A_TILE), db_lo = make_smem_desc(sb + C::B_TILE);
#pragma unroll
                  for (int k = 0; k < KSTEPS; ++k) {
                    if (k < nk) {
                      const uint64_t koff = (uint64_t)((k * UMMA_K_BYTES) >> 4);
                      umma_pair<KIND>(da_lo + koff, db_hi + koff, tmem_d, idesc, (ks > ks0 || k > 0) ? 1u : 0u);
                      umma_pair<KIND>(da_hi + koff, db_lo + koff, tmem_d, idesc, 1u);
                    }
                  }
                }
#pragma unroll
                for (int k = 0; k < KSTEPS; ++k) {
                  if (k < nk) {
                    const uint64_t koff = (uint64_t)((k * UMMA_K_BYTES) >> 4);
                    umma_pair<KIND>(da_hi + koff, db_hi + koff, tmem_d, idesc, (NTERMS == 3 || ks > ks0 || k > 0) ? 1u : 0u);
                  }
                }
                umma_commit_pair(empty_bar(stage));                  // slot free in both CTAs once these MMAs retire
                if (ks == ks1 - 1) umma_commit_pair(tfull_bar(acc));  // accumulation chain complete (both CTAs)
              }
              if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            }
          }
          ks0 = ks1;
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue warps (TMEM lane quarter = warp % 4; column half = (warp-4)/4) ======
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
    const uint32_t stage_u32 = epi_base + (warp - FIRST_EPI_WARP) * (STAGE_EPI_BYTES + (C::INBOX ? INBOX_BYTES : 0));
    uint8_t* stage = smem_gen + (stage_u32 - smem_base);

    const uint32_t tempty_leader = mapa(tempty_bar(0), 0);
    if (C::HALF0 == C::HALF1)     // one copy of the epilogue code serves both column halves
      epilogue_loop<C, C::HALF0, SPLITK>(warp < FIRST_EPI_WARP + 4 ? 0 : C::HALF0, warp & 3, lane, rank, tmem_base, tfull_bar(0),
                                 tempty_leader, stage, stage_u32, n_tiles, n_blocks, k_slabs, split_k, split_per, chunk_slabs, lead_chains, M, N, ep, path_flags, smaps);
    else if (warp < FIRST_EPI_WARP + 4)
      epilogue_loop<C, C::HALF0, SPLITK>(0, warp & 3, lane, rank, tmem_base, tfull_bar(0), tempty_leader, stage, stage_u32, n_tiles,
                                 n_blocks, k_slabs, split_k, split_per, chunk_slabs, lead_chains, M, N, ep, path_flags, smaps);
    else
      epilogue_loop<C, C::HALF1, SPLITK>(C::HALF0, warp & 3, lane, rank, tmem_base, tfull_bar(0), tempty_leader, stage, stage_u32,
                                 n_tiles, n_blocks, k_slabs, split_k, split_per, chunk_slabs, lead_chains, M, N, ep, path_flags, smaps);
  }

  tcgen05_fence_before();
  cluster_sync_all();   // the peer may still signal our barriers / read our smem through the MMA until here
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(C::TMEM_COLS) : "memory");
  }
}

}  // namespace tc2

// host side ---------------------------------------------------------------------------------------
// test hook (usf_debug_set_store_path): 4 = always the register/patch store path, 32 = the epilogue warps store their
// staged boxes themselves (no TMA stores), 256 = the kernel reads the coupling residual lane-per-row (no in-box)
extern int g_store_path;

// 3xTF32 engine: K-slabs (32 elements each) accumulated in TMEM before the partial tile is added into fp32 registers with
// round-to-nearest (the tensor core truncates when it accumulates: long chains carry a systematic toward-zero bias).  The
// fp16-split engine closes a chain every slab (the kernel's rule); the single-pass engines accumulate the whole K.
constexpr int CHUNK_SLABS = 2;
// fp16-split engine: the first LEAD_CHAINS accumulation chains of every tile span twice the K-slabs, so the tensor core keeps
// running on the next tile while the epilogue warps still store the previous one (two TMEM accumulators = two chains of
// run-ahead).  Not for 3xTF32: its chains already hold 48 MMA steps, and the toward-zero bias of longer chains shows in
// the gradients.
constexpr int LEAD_CHAINS = 2;

// fp16 output plane [rows, cols] (row pitch ld halves) for the TMA store path: box = 32 rows x box_cols (32: 64B swizzle,
// 16: 32B swizzle) columns
inline int make_store_map16(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld, int box_cols) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return fail(USF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available%s%s");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B,
                   CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled (store map) failed with CUresult %d (rows=%lld cols=%lld ld=%lld)",
             (int)r, rows, cols, ld);
    return USF_ERR_CUDA;
  }
  return USF_OK;
}

// fp32 output plane [rows, cols] for the TMA store path: box = 32 rows x 16 columns (64-byte rows, 64B swizzle)
inline int make_store_map32(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return fail(USF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available%s%s");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {16, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled (fp32 store map) failed with CUresult %d (rows=%lld cols=%lld ld=%lld)",
             (int)r, rows, cols, ld);
    return USF_ERR_CUDA;
  }
  return USF_OK;
}

template <int BLOCK_N, int NTERMS, int KIND, bool SPLITK = false>
int launch_gemm_tc2_cfg(const usf_linear_args* a, const Epilogue& ep_in, cudaStream_t st) {
  using C = tc2::Config<BLOCK_N, NTERMS, KIND>;
  constexpr bool F16S = NTERMS == 3 && KIND == tc2::KIND_F16;
  // split-K exists for the fp16-split engine (the training pass); every other engine runs the plain kernel
  if (!SPLITK && F16S && a->split_k > 1)
    return launch_gemm_tc2_cfg<BLOCK_N, NTERMS, KIND, F16S>(a, ep_in, st);
  static bool attr_set_dev[MAX_DEVICES] = {false};
  bool& attr_set = attr_set_dev[current_device_slot()];
  auto kern = tc2::gemm_tc2_kernel<BLOCK_N, NTERMS, KIND, SPLITK>;
  const int dt = KIND == tc2::KIND_TF32 ? 0 : KIND == tc2::KIND_BF16 ? 1 : 2;
  if (!attr_set) {
    USF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  CUtensorMap ma, mal, mw, mwl;
  int rc;
  if ((rc = make_operand_map(&ma, a->a, a->M, a->K, a->lda, tc::BLOCK_M, dt))) return rc;
  if ((rc = make_operand_map(&mw, a->w, a->N, a->K, a->ldw, C::HALF_N, dt))) return rc;
  if (NTERMS == 3) {
    if ((rc = make_operand_map(&mal, a->a_lo, a->M, a->K, a->lda, tc::BLOCK_M, dt))) return rc;
    if ((rc = make_operand_map(&mwl, a->w_lo, a->N, a->K, a->ldw, C::HALF_N, dt))) return rc;
  } else {
    mal = ma;
    mwl = mw;
  }
  // aligned output planes (16-byte aligned, pitch a 16-byte multiple, N a multiple of 8) leave through the staged,
  // coalesced store path; anything else through the generic register/patch path
  Epilogue ep = ep_in;
  ep.fast_store = (ep.vec_ok && a->N % 8 == 0 && !(g_store_path & 4)) ? 1 : 0;
  ep.async_store = (ep.fast_store && !(g_store_path & 32) && ep.out_h16 && !ep.out_f32 && !ep.out_hi && !ep.out_bf16 &&
                    !ep.colscale && !ep.postsub && !ep.resid_hi) ? 1 : 0;
  // mode 2: bf16 and / or fp32 planes (bf16 / tf32 precision modes), fp32 residual allowed
  if (!ep.async_store && ep.fast_store && !(g_store_path & 32) && !ep.out_h16 && !ep.out_hi && (ep.out_bf16 || ep.out_f32) &&
      !ep.colscale && !ep.postsub && !ep.resid_h16 && !(SPLITK && a->split_k > 1))
    ep.async_store = 2;
  tc2::StoreMaps sm;
  memset(&sm, 0, sizeof(sm));
  if (ep.async_store == 2) {
    if (ep.out_bf16) {
      if ((rc = make_store_map16(&sm.h32, ep.out_bf16, a->M, a->N, ep.ld_bf16, 32))) return rc;
      if ((rc = make_store_map16(&sm.h16, ep.out_bf16, a->M, a->N, ep.ld_bf16, 16))) return rc;
    }
    if (ep.out_f32 && (rc = make_store_map32(&sm.l32, ep.out_f32, a->M, a->N, ep.ld_f32))) return rc;
  } else if (ep.async_store) {
    if ((rc = make_store_map16(&sm.h32, ep.out_h16, a->M, a->N, ep.ld_16, 32))) return rc;
    if ((rc = make_store_map16(&sm.l32, ep.out_l16, a->M, a->N, ep.ld_16, 32))) return rc;
    if ((rc = make_store_map16(&sm.h16, ep.out_h16, a->M, a->N, ep.ld_16, 16))) return rc;
    if ((rc = make_store_map16(&sm.l16, ep.out_l16, a->M, a->N, ep.ld_16, 16))) return rc;
  }
  // split-K (training: dW = dY^T . X): the K-slabs of a tile are cut into `split_k` work items that add their partial tiles
  // into the fp32 output (red.global.add.v4.f32); the caller zeroes / pre-loads the output (usf_linear does, see capi.cu)
  int split_k = 1, split_per = 0;
  if (SPLITK && a->split_k > 1) {
    const int k_slabs = (int)((a->K + C::ELEMS_PER_SLAB - 1) / C::ELEMS_PER_SLAB);
    const int per = (k_slabs + a->split_k - 1) / a->split_k;   // (an accumulation chain of this engine is one slab)
    split_k = (k_slabs + per - 1) / per;                    // every work item gets at least one slab
    split_per = per;
    USF_REQUIRE(ep.fast_store && ep.out_f32 && !ep.out_h16 && !ep.out_hi && !ep.out_bf16 && !ep.bias && !ep.relu &&
                    !ep.resid_hi && !ep.resid_h16 && !ep.colscale && !ep.postsub,
                "split_k > 1 accumulates plain partial products into an aligned fp32 output (no other epilogue feature)");
    ep.atomic_out = split_k > 1 ? 1 : 0;
  }
  const long long tiles = ((a->M + 2 * tc::BLOCK_M - 1) / (2 * tc::BLOCK_M)) * ((a->N + BLOCK_N - 1) / BLOCK_N) * split_k;
  const int pairs = num_sms() / 2;
  const int grid = 2 * (int)(tiles < pairs ? tiles : pairs);
  USF_CUDA_OK(launch_chain(kern, dim3(grid), dim3(tc::NUM_THREADS), (size_t)C::SMEM_BYTES, st, ma, mal, mw, mwl, (long long)a->M,
                           (int)a->N, (int)a->K, NTERMS == 3 ? CHUNK_SLABS : 0,
                           (NTERMS == 3 && KIND == tc2::KIND_F16) ? LEAD_CHAINS : 0, split_k, split_per, ep, sm, g_store_path));
  return USF_OK;
}

// BLOCK_N choice for the pair kernel: least padded MMA work, ties to the wider tile
inline int pick_block_n2(int N) {
  static const int cands[] = {256, 208, 128, 64, 32};
  int best = 256;
  double best_cost = 1e30;
  for (int bn : cands) {
    int nb = (N + bn - 1) / bn;
    double waste = (double)nb * bn / N;
    double cost = waste * (1.0 + 0.25 * 128.0 / bn) * (1.0 + 0.01 * nb);  // narrow tiles re-read A more often
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

template <int NTERMS, int KIND>
int launch_gemm_tc2_terms(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st, int bn) {
  switch (bn) {
    case 256: return launch_gemm_tc2_cfg<256, NTERMS, KIND>(a, ep, st);
    case 208: return launch_gemm_tc2_cfg<208, NTERMS, KIND>(a, ep, st);
    case 128: return launch_gemm_tc2_cfg<128, NTERMS, KIND>(a, ep, st);
    case 64: return launch_gemm_tc2_cfg<64, NTERMS, KIND>(a, ep, st);
    case 32: return launch_gemm_tc2_cfg<32, NTERMS, KIND>(a, ep, st);
  }
  return fail(USF_ERR_INVALID, "unsupported BLOCK_N (built: 256, 208, 128, 64, 32)%s%s");
}

int launch_gemm_tc2_3xtf32(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st, int bn);
int launch_gemm_tc2_tf32(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st, int bn);
int launch_gemm_tc2_bf16(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st, int bn);
int launch_gemm_tc2_3xf16(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st, int bn);

extern int g_force_block_n;   // test hook (usf_debug_set_block_n)

inline int launch_gemm_tc(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st) {
  if (a->M == 0 || a->N == 0) return USF_OK;
  const bool two_byte = a->engine == USF_ENGINE_TC_BF16 || a->engine == USF_ENGINE_TC_3XF16;
  const int kmul = two_byte ? 8 : 4;
  USF_REQUIRE(a->K > 0, "K must be positive");
  USF_REQUIRE(a->M < (1LL << 31) - 512, "tcgen05 engine: M must fit a TMA coordinate");
  USF_REQUIRE(aligned16(a->a) && aligned16(a->w) && a->lda % kmul == 0 && a->ldw % kmul == 0,
              "tcgen05 engines need 16-byte aligned operands and 16-byte multiples for lda/ldw");
  USF_REQUIRE(!a->trans_w, "trans_w is a SIMT-engine option");
  if (a->engine == USF_ENGINE_TC_3XTF32 || a->engine == USF_ENGINE_TC_3XF16)
    USF_REQUIRE(a->a_lo && a->w_lo && aligned16(a->a_lo) && aligned16(a->w_lo), "split engines need a_lo and w_lo planes");
  const int bn = g_force_block_n > 0 ? g_force_block_n : pick_block_n2(a->N);
  if (a->engine == USF_ENGINE_TC_3XF16) return launch_gemm_tc2_3xf16(a, ep, st, bn);
  if (a->engine == USF_ENGINE_TC_3XTF32) return launch_gemm_tc2_3xtf32(a, ep, st, bn);
  if (a->engine == USF_ENGINE_TC_TF32) return launch_gemm_tc2_tf32(a, ep, st, bn);
  return launch_gemm_tc2_bf16(a, ep, st, bn);
}

}  // namespace usf
