// C ABI of libusflows_b200.so (see include/usflows_b200.h for the contract of every entry point).
#include "common.cuh"
#include "conditioner.cuh"
#include "conv_tc.cuh"
#include "elementwise.cuh"
#include "flow_small.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc2.cuh"
#include "image.cuh"
#include "prep.cuh"
#include "radial.cuh"
#include "train.cuh"
#include "plan.cuh"

namespace usf {
// csrc/conv_pix.cuh (compiled in conv_pix_inst.cu only: the kernel is not a template)
int launch_conv_pix(const usf_conv_pix_args* a, cudaStream_t st);
int launch_pix_encode(const float* x, long long ldx, long long rows, int c, int hw, const float* mask, int relu, void* out16,
                      int* overflow_flag, cudaStream_t st);
}  // namespace usf

namespace usf {

thread_local char g_err[512] = "";
int g_force_block_n = 0;
int g_store_path = 0;
int g_use_pdl = 1;

int num_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

int make_epilogue(const usf_linear_args* a, Epilogue* ep) {
  USF_REQUIRE(a->out_f32 || a->out_hi || a->out_bf16 || a->out_h16, "usf_linear needs at least one output plane");
  USF_REQUIRE((a->out_hi == nullptr) == (a->out_lo == nullptr), "out_hi and out_lo come as a pair");
  USF_REQUIRE(!a->resid_lo || a->resid, "resid_lo without resid");
  ep->bias = a->bias;
  ep->resid_hi = a->resid;
  ep->resid_lo = a->resid_lo;
  ep->colscale = a->colscale;
  ep->postsub = a->postsub;
  ep->out_f32 = a->out_f32;
  ep->out_hi = a->out_hi;
  ep->out_lo = a->out_lo;
  ep->out_bf16 = reinterpret_cast<__nv_bfloat16*>(a->out_bf16);
  ep->ldr = a->ldr;
  ep->ld_f32 = a->ld_f32;
  ep->ld_split = a->ld_split;
  ep->ld_bf16 = a->ld_bf16;
  ep->resid_sign = a->resid_sign;
  ep->relu = a->relu;
  USF_REQUIRE((a->out_h16 == nullptr) == (a->out_l16 == nullptr), "out_h16 and out_l16 come as a pair");
  USF_REQUIRE((a->resid_h16 == nullptr) == (a->resid_l16 == nullptr), "resid_h16 and resid_l16 come as a pair");
  USF_REQUIRE(!(a->resid && a->resid_h16), "give the residual either as fp32 planes or as fp16 split planes");
  ep->resid_h16 = reinterpret_cast<const __half*>(a->resid_h16);
  ep->resid_l16 = reinterpret_cast<const __half*>(a->resid_l16);
  ep->out_h16 = reinterpret_cast<__half*>(a->out_h16);
  ep->out_l16 = reinterpret_cast<__half*>(a->out_l16);
  ep->ldr_16 = a->ldr_16;
  ep->ld_16 = a->ld_16;
  ep->overflow_flag = a->overflow_flag;
  bool ok = true;
  if (a->resid_h16) ok = ok && aligned16(a->resid_h16) && aligned16(a->resid_l16) && a->ldr_16 % 8 == 0;
  if (a->out_h16) ok = ok && aligned16(a->out_h16) && aligned16(a->out_l16) && a->ld_16 % 8 == 0;
  if (a->bias) ok = ok && aligned16(a->bias);
  if (a->colscale) ok = ok && aligned16(a->colscale);
  if (a->postsub) ok = ok && aligned16(a->postsub);
  if (a->resid) ok = ok && aligned16(a->resid) && a->ldr % 4 == 0;
  if (a->resid_lo) ok = ok && aligned16(a->resid_lo);
  if (a->out_f32) ok = ok && aligned16(a->out_f32) && a->ld_f32 % 4 == 0;
  if (a->out_hi) ok = ok && aligned16(a->out_hi) && aligned16(a->out_lo) && a->ld_split % 4 == 0;
  if (a->out_bf16) ok = ok && aligned16(a->out_bf16) && a->ld_bf16 % 8 == 0;
  ep->vec_ok = ok ? 1 : 0;
  ep->fast_store = 0;  // set by the pair-kernel launcher
  ep->async_store = 0;
  ep->atomic_out = 0;
  return USF_OK;
}

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

static OutPlanes to_out_planes(const usf_planes* p, int32_t* overflow_flag) {
  OutPlanes o{nullptr, nullptr, nullptr, nullptr, 0, 0, 0};
  if (!p) return o;
  o.f32 = p->f32; o.ld_f32 = p->ld_f32;
  o.hi = p->hi; o.lo = p->lo; o.ld_split = p->ld_split;
  o.bf16 = reinterpret_cast<__nv_bfloat16*>(p->bf16); o.ld_bf16 = p->ld_bf16;
  o.h16 = reinterpret_cast<__half*>(p->h16); o.l16 = reinterpret_cast<__half*>(p->l16); o.ld_16 = p->ld_16;
  o.overflow_flag = overflow_flag;
  return o;
}

static inline DrawCtr to_draw(const usf_draw* d) {
  return DrawCtr{(unsigned long long)d->seed, (unsigned long long)d->offset, (long long)d->row0,
                 reinterpret_cast<const long long*>(d->dev_params)};
}

static inline bool dequant_ok(const usf_dequant* dq) {
  return dq && (dq->mode == USF_DEQUANT_UNIFORM || dq->mode == USF_DEQUANT_MIDPOINT);
}

// Scope in which this thread's stream-capture interaction mode is "relaxed", so an allocation / release issued while the
// thread happens to be capturing a CUDA graph neither fails nor invalidates the capture.
struct RelaxedCaptureMode {
  cudaStreamCaptureMode mode = cudaStreamCaptureModeRelaxed;
  RelaxedCaptureMode() { cudaThreadExchangeStreamCaptureMode(&mode); }
  ~RelaxedCaptureMode() { cudaThreadExchangeStreamCaptureMode(&mode); }
};

}  // namespace usf

using namespace usf;

extern "C" {

const char* usf_last_error(void) { return g_err; }
int usf_abi_version(void) { return USF_ABI_VERSION; }

int usf_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes) {
  int dev = 0;
  USF_CUDA_OK(cudaGetDevice(&dev));
  int v = 0;
  if (sm_count) { USF_CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev)); *sm_count = v; }
  if (cc_major) { USF_CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev)); *cc_major = v; }
  if (cc_minor) { USF_CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev)); *cc_minor = v; }
  if (l2_bytes) { USF_CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, dev)); *l2_bytes = v; }
  return USF_OK;
}

int usf_debug_set_block_n(int bn) {  // test hook: force the tcgen05 tile width (0 = automatic)
  g_force_block_n = bn;
  return USF_OK;
}

int usf_debug_set_store_path(int flags) {  // test hook: force the contraction's other store / residual paths (0 = automatic)
  USF_REQUIRE((flags & ~(4 | 32 | 256)) == 0, "store path flags: 4, 32, 256 or a combination");
  g_store_path = flags;
  return USF_OK;
}

int usf_debug_set_pdl(int on) {  // test hook: programmatic dependent launch of the kernel chain (default on)
  g_use_pdl = on ? 1 : 0;
  return USF_OK;
}

int usf_linear(const usf_linear_args* a, void* stream) {
  USF_REQUIRE(a != nullptr, "null args");
  USF_REQUIRE(a->M >= 0 && a->N >= 0 && a->K >= 0, "negative extent");
  USF_REQUIRE(a->a && a->w, "null operand");
  Epilogue ep;
  int rc = make_epilogue(a, &ep);
  if (rc) return rc;
  switch (a->engine) {
    case USF_ENGINE_SIMT: return launch_gemm_simt(a, ep, S(stream));
    case USF_ENGINE_TC_3XTF32:
    case USF_ENGINE_TC_TF32:
    case USF_ENGINE_TC_BF16:
    case USF_ENGINE_TC_3XF16:
      if (a->split_k > 1 && a->engine == USF_ENGINE_TC_3XF16 && a->M > 0 && a->N > 0)   // partial tiles are added: start from zero
        USF_CUDA_OK(cudaMemset2DAsync(a->out_f32, (size_t)a->ld_f32 * 4, 0, (size_t)a->N * 4, (size_t)a->M, S(stream)));
      return launch_gemm_tc(a, ep, S(stream));
  }
  return fail(USF_ERR_INVALID, "unknown engine%s%s");
}

int usf_flow_small(const float* x, int64_t ldx, int64_t rows, int32_t d, const int32_t* prog, int32_t n_ops,
                   const float* blob, int32_t blob_floats, int32_t D, int32_t H, float* out, int64_t ldo, void* stream) {
  USF_REQUIRE(x && prog && blob && out && rows >= 0 && n_ops >= 0 && blob_floats > 0, "bad input");
  return launch_flow_small(x, ldx, rows, d, prog, n_ops, blob, blob_floats, D, H, out, ldo, S(stream));
}

int usf_ingest(const float* x, int64_t ldx, int64_t rows, int32_t d, const float* dv, const float* mul,
               const float* sub, float* out_f32, int64_t ld_f32, float* out_hi, float* out_lo, int64_t ld_split,
               void* out_bf16, int64_t ld_bf16, void* stream) {
  USF_REQUIRE(x && rows >= 0 && d > 0, "bad input");
  USF_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), "out_hi and out_lo come as a pair");
  if (rows == 0) return USF_OK;
  OutPlanes o{out_f32, out_hi, out_lo, reinterpret_cast<__nv_bfloat16*>(out_bf16), ld_f32, ld_split, ld_bf16};
  const bool vec = planes_vec_ok(o) && aligned16(x) && ldx % 4 == 0 && d % 4 == 0 && (!dv || aligned16(dv)) &&
                   (!mul || aligned16(mul)) && (!sub || aligned16(sub)) && (!out_bf16 || d % 8 == 0 || true);
  if (vec)
    USF_CUDA_OK(launch_chain(ingest_kernel<true, LoadF32>, dim3(ew_grid(rows * (d / 4), 256)), dim3(256), 0, S(stream), LoadF32{x, (long long)ldx}, (long long)rows, (int)d, dv, mul, sub, o));
  else
    USF_CUDA_OK(launch_chain(ingest_kernel<false, LoadF32>, dim3(ew_grid(rows * d, 256)), dim3(256), 0, S(stream), LoadF32{x, (long long)ldx}, (long long)rows, (int)d, dv, mul, sub, o));
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_ingest_f16(const float* x, int64_t ldx, int64_t rows, int32_t d, const float* dv, const float* mul,
                   const float* sub, void* out_h16, void* out_l16, int64_t ld_16, int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(x && rows >= 0 && d > 0 && out_h16 && out_l16, "bad input");
  if (rows == 0) return USF_OK;
  OutPlanes o{nullptr, nullptr, nullptr, nullptr, 0, 0, 0};
  o.h16 = reinterpret_cast<__half*>(out_h16);
  o.l16 = reinterpret_cast<__half*>(out_l16);
  o.ld_16 = ld_16;
  o.overflow_flag = overflow_flag;
  const bool vec = planes_vec_ok(o) && aligned16(x) && ldx % 4 == 0 && d % 4 == 0 && (!dv || aligned16(dv)) &&
                   (!mul || aligned16(mul)) && (!sub || aligned16(sub));
  if (vec)
    USF_CUDA_OK(launch_chain(ingest_kernel<true, LoadF32>, dim3(ew_grid(rows * (d / 4), 256)), dim3(256), 0, S(stream), LoadF32{x, (long long)ldx}, (long long)rows, (int)d, dv, mul, sub, o));
  else
    USF_CUDA_OK(launch_chain(ingest_kernel<false, LoadF32>, dim3(ew_grid(rows * d, 256)), dim3(256), 0, S(stream), LoadF32{x, (long long)ldx}, (long long)rows, (int)d, dv, mul, sub, o));
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_ingest_u8(const uint8_t* x, int64_t ldx, int64_t rows, int32_t d, const usf_dequant* dq, const float* dv,
                  const float* mul, const float* sub, const usf_planes* out, int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(x && out && rows >= 0 && d > 0 && ldx >= d, "bad input");
  USF_REQUIRE(dequant_ok(dq), "bad dequantisation (null, or mode not USF_DEQUANT_UNIFORM / USF_DEQUANT_MIDPOINT)");
  USF_REQUIRE((out->hi == nullptr) == (out->lo == nullptr) && (out->h16 == nullptr) == (out->l16 == nullptr), "planes come as pairs");
  USF_REQUIRE(out->f32 || out->hi || out->bf16 || out->h16, "usf_ingest_u8 needs an output plane");
  if (rows == 0) return USF_OK;
  const OutPlanes o = to_out_planes(out, overflow_flag);
  const LoadU8 in{x, (long long)ldx, (unsigned long long)dq->seed, (long long)dq->row0,
                  reinterpret_cast<const long long*>(dq->dev_params), (int)dq->mode};
  const bool vec = planes_vec_ok(o) && (reinterpret_cast<uintptr_t>(x) & 3u) == 0 && ldx % 4 == 0 && d % 4 == 0 &&
                   (!dv || aligned16(dv)) && (!mul || aligned16(mul)) && (!sub || aligned16(sub));
  if (vec)
    USF_CUDA_OK(launch_chain(ingest_kernel<true, LoadU8>, dim3(ew_grid(rows * (d / 4), 256)), dim3(256), 0, S(stream), in, (long long)rows, (int)d, dv, mul, sub, o));
  else
    USF_CUDA_OK(launch_chain(ingest_kernel<false, LoadU8>, dim3(ew_grid(rows * d, 256)), dim3(256), 0, S(stream), in, (long long)rows, (int)d, dv, mul, sub, o));
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_base_logprob(const float* z, const float* z_lo, int64_t ldz, int64_t rows, int32_t d, const float* loc,
                     const float* scale, int32_t base_kind, float add_const, float* out, void* stream) {
  USF_REQUIRE(z && loc && scale && out && d > 0 && rows >= 0, "bad input");
  USF_REQUIRE(base_kind == USF_BASE_LAPLACE || base_kind == USF_BASE_NORMAL, "unknown base distribution");
  if (rows == 0) return USF_OK;
  const bool vec = aligned16(z) && (!z_lo || aligned16(z_lo)) && ldz % 4 == 0 && d % 4 == 0 && aligned16(loc) && aligned16(scale);
  const int grid = ew_grid(rows * 32, BLP_THREADS);
  if (vec)
    USF_CUDA_OK(launch_chain(base_logprob_kernel<true>, dim3(grid), dim3(BLP_THREADS), 0, S(stream), z, z_lo, (long long)ldz, (long long)rows, (int)d, loc, scale, (int)base_kind, add_const, out));
  else
    USF_CUDA_OK(launch_chain(base_logprob_kernel<false>, dim3(grid), dim3(BLP_THREADS), 0, S(stream), z, z_lo, (long long)ldz, (long long)rows, (int)d, loc, scale, (int)base_kind, add_const, out));
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_base_sample(int64_t rows, int32_t d, const float* loc, const float* scale, int32_t base_kind, uint64_t seed,
                    uint64_t offset, float* out_f32, int64_t ld_f32, float* out_hi, float* out_lo, int64_t ld_split,
                    void* out_bf16, int64_t ld_bf16, void* stream) {
  const usf_draw dr{seed, offset, 0, nullptr};
  return usf_base_sample_at(rows, d, loc, scale, base_kind, &dr, out_f32, ld_f32, out_hi, out_lo, ld_split, out_bf16, ld_bf16,
                            stream);
}

int usf_base_sample_at(int64_t rows, int32_t d, const float* loc, const float* scale, int32_t base_kind, const usf_draw* draw,
                       float* out_f32, int64_t ld_f32, float* out_hi, float* out_lo, int64_t ld_split, void* out_bf16,
                       int64_t ld_bf16, void* stream) {
  USF_REQUIRE(loc && scale && d > 0 && rows >= 0, "bad input");
  USF_REQUIRE(draw && draw->row0 >= 0, "bad draw (null, or negative row0)");
  USF_REQUIRE(base_kind == USF_BASE_LAPLACE || base_kind == USF_BASE_NORMAL, "unknown base distribution");
  USF_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), "out_hi and out_lo come as a pair");
  if (rows == 0) return USF_OK;
  OutPlanes o{out_f32, out_hi, out_lo, reinterpret_cast<__nv_bfloat16*>(out_bf16), ld_f32, ld_split, ld_bf16};
  const int vec = planes_vec_ok(o) ? 1 : 0;
  base_sample_kernel<<<ew_grid(rows * ((d + 3) / 4), 256), 256, 0, S(stream)>>>(rows, d, loc, scale, base_kind, to_draw(draw), o, vec);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_quantize_u8(const float* y, int64_t ldy, int64_t rows, int32_t d, uint8_t* out, int64_t ldo, void* stream) {
  USF_REQUIRE(y && out && rows >= 0 && d > 0 && ldy >= d && ldo >= d, "bad input");
  if (rows == 0) return USF_OK;
  const bool vec = aligned16(y) && ldy % 4 == 0 && d % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0 && ldo % 4 == 0;
  if (vec)
    quantize_u8_kernel<true><<<ew_grid(rows * (d / 4), 256), 256, 0, S(stream)>>>(y, ldy, rows, d, out, ldo);
  else
    quantize_u8_kernel<false><<<ew_grid(rows * d, 256), 256, 0, S(stream)>>>(y, ldy, rows, d, out, ldo);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_affine_couple(const float* st, int64_t ld_st, int64_t rows, int32_t h, float* x_f32, int64_t ld_f32, float* x_hi,
                      float* x_lo, int64_t ld_split, void* x_bf16, int64_t ld_bf16, void* x_h16, void* x_l16, int64_t ld_16,
                      int32_t* overflow_flag, float direction, float s_min, float s_max, float* row_ladj, void* stream) {
  USF_REQUIRE(st && rows >= 0 && h > 0, "bad input");
  USF_REQUIRE(x_f32 || x_hi || x_bf16 || x_h16, "usf_affine_couple needs the planes of x");
  USF_REQUIRE((x_hi == nullptr) == (x_lo == nullptr) && (x_h16 == nullptr) == (x_l16 == nullptr), "planes come as pairs");
  USF_REQUIRE(direction == 1.f || direction == -1.f, "direction must be +1 or -1");
  if (rows == 0) return USF_OK;
  XPlanes p{x_f32, x_hi, x_lo, reinterpret_cast<__nv_bfloat16*>(x_bf16), reinterpret_cast<__half*>(x_h16),
            reinterpret_cast<__half*>(x_l16), ld_f32, ld_split, ld_bf16, ld_16, overflow_flag};
  affine_couple_kernel<<<ew_grid(rows * 32, 256), 256, 0, S(stream)>>>(st, ld_st, rows, h, p, direction, s_min, s_max, row_ladj);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_radial_logprob(const float* z, const float* z_lo, int64_t ldz, int64_t rows, int32_t d, const float* loc,
                       int32_t p_kind, int32_t norm_kind, const float* norm_params, int32_t n_comp, float dv_const,
                       float add_const, float* out, void* stream) {
  USF_REQUIRE(z && loc && norm_params && out && d > 0 && rows >= 0, "bad input");
  USF_REQUIRE(p_kind == USF_LP_INF || p_kind == USF_LP_1 || p_kind == USF_LP_2, "p must be 1, 2 or inf");
  USF_REQUIRE(norm_kind == USF_NORM_LOGNORMAL ||
              (norm_kind >= USF_NORM_GAMMA_MIXTURE && norm_kind <= USF_NORM_LOGNORMAL_MIXTURE && n_comp >= 1 && n_comp <= RAD_MAX_COMP),
              "unknown norm distribution / too many mixture components");
  if (rows == 0) return USF_OK;
  const bool vec = aligned16(z) && (!z_lo || aligned16(z_lo)) && ldz % 4 == 0 && d % 4 == 0 && aligned16(loc);
  const int grid = ew_grid(rows * 32, RAD_THREADS);
  if (vec)
    radial_logprob_kernel<true><<<grid, RAD_THREADS, 0, S(stream)>>>(z, z_lo, ldz, rows, d, loc, p_kind, norm_kind, norm_params, n_comp, dv_const, add_const, out);
  else
    radial_logprob_kernel<false><<<grid, RAD_THREADS, 0, S(stream)>>>(z, z_lo, ldz, rows, d, loc, p_kind, norm_kind, norm_params, n_comp, dv_const, add_const, out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_radial_sample(int64_t rows, int32_t d, const float* loc, int32_t p_kind, int32_t norm_kind,
                      const float* norm_params, int32_t n_comp, uint64_t seed, uint64_t offset, float* out, int64_t ldo,
                      void* stream) {
  const usf_draw dr{seed, offset, 0, nullptr};
  return usf_radial_sample_at(rows, d, loc, p_kind, norm_kind, norm_params, n_comp, &dr, out, ldo, stream);
}

int usf_radial_sample_at(int64_t rows, int32_t d, const float* loc, int32_t p_kind, int32_t norm_kind,
                         const float* norm_params, int32_t n_comp, const usf_draw* draw, float* out, int64_t ldo,
                         void* stream) {
  USF_REQUIRE(loc && norm_params && out && d > 0 && rows >= 0 && ldo >= d, "bad input");
  USF_REQUIRE(draw && draw->row0 >= 0, "bad draw (null, or negative row0)");
  USF_REQUIRE(p_kind == USF_LP_INF || p_kind == USF_LP_1 || p_kind == USF_LP_2, "p must be 1, 2 or inf");
  USF_REQUIRE(norm_kind == USF_NORM_LOGNORMAL ||
              (norm_kind >= USF_NORM_GAMMA_MIXTURE && norm_kind <= USF_NORM_LOGNORMAL_MIXTURE && n_comp >= 1 && n_comp <= RAD_MAX_COMP),
              "unknown norm distribution / too many mixture components");
  if (rows == 0) return USF_OK;
  radial_sample_kernel<<<ew_grid(rows * 32, RAD_THREADS), RAD_THREADS, 0, S(stream)>>>(rows, d, loc, p_kind, norm_kind, norm_params, n_comp, to_draw(draw), out, ldo);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_gate_norm(const float* o, int64_t ldo, const float* xres, int64_t ldx, int64_t rows, int32_t n, int32_t gated,
                  int32_t pre_relu, const float* gamma, const float* beta, float eps, float* y_f32, int64_t ldy, const usf_planes* act,
                  int32_t act_relu, const usf_planes* raw, int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(o && rows >= 0 && n > 0 && n <= 6144, "bad input (n must be in 1..6144)");
  USF_REQUIRE(!gated || xres, "a gated update needs the residual stream");
  USF_REQUIRE((gamma == nullptr) == (beta == nullptr), "gamma and beta come as a pair");
  USF_REQUIRE(y_f32 || act || raw, "usf_gate_norm needs at least one output");
  if (act) USF_REQUIRE((act->hi == nullptr) == (act->lo == nullptr) && (act->h16 == nullptr) == (act->l16 == nullptr), "planes come as pairs");
  if (raw) USF_REQUIRE((raw->hi == nullptr) == (raw->lo == nullptr) && (raw->h16 == nullptr) == (raw->l16 == nullptr), "planes come as pairs");
  if (rows == 0) return USF_OK;
  const OutPlanes a = to_out_planes(act, overflow_flag), rw = to_out_planes(raw, overflow_flag);
  bool vec = n % 4 == 0 && aligned16(o) && ldo % 4 == 0 && (!gated || (aligned16(xres) && ldx % 4 == 0)) &&
             (!gamma || (aligned16(gamma) && aligned16(beta))) && (!y_f32 || (aligned16(y_f32) && ldy % 4 == 0));
  if (act) vec = vec && planes_vec_ok(a);
  if (raw) vec = vec && planes_vec_ok(rw);
  // lanes per row: enough to cover the row once (4 elements per lane on the vector path), at least 4, at most a warp
  const int per_lane = vec ? 4 : 1;
  int G = 4;
  while (G < 32 && G * per_lane < n) G *= 2;
  const size_t smem = (size_t)(GN_THREADS / 32) * (32 / G) * n * sizeof(float);
  const int grid = ew_grid(rows * G, GN_THREADS);
  void (*kern)(const float*, long long, const float*, long long, long long, int, int, int, const float*, const float*, float,
               float*, long long, OutPlanes, int, int, OutPlanes, int) = nullptr;
  if (vec) kern = G == 4 ? gate_norm_kernel<true, 4> : G == 8 ? gate_norm_kernel<true, 8> : G == 16 ? gate_norm_kernel<true, 16> : gate_norm_kernel<true, 32>;
  else kern = G == 4 ? gate_norm_kernel<false, 4> : G == 8 ? gate_norm_kernel<false, 8> : G == 16 ? gate_norm_kernel<false, 16> : gate_norm_kernel<false, 32>;
  if (smem > 48 * 1024) USF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, GN_THREADS, smem, S(stream)>>>(o, ldo, xres, ldx, rows, n, gated ? 1 : 0, pre_relu ? 1 : 0, gamma, beta, eps, y_f32, ldy, a,
                                             act ? 1 : 0, act_relu ? 1 : 0, rw, raw ? 1 : 0);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_layout_transpose(const float* in, int64_t n, int32_t a, int32_t b, const float* scale, int32_t scale_mode,
                         int32_t scale_on_input, float* out, void* stream) {
  USF_REQUIRE(in && out && n >= 0 && a > 0 && b > 0, "bad input");
  USF_REQUIRE(scale_mode >= 0 && scale_mode <= 2 && (scale_mode == 0 || scale), "scale_mode 0 (none), 1 (multiply) or 2 (divide)");
  if (n == 0) return USF_OK;
  const long long tiles = (long long)n * ((a + 31) / 32) * ((b + 31) / 32);
  layout_kernel<float><<<ew_grid(tiles * 256, 256), 256, 0, S(stream)>>>(in, n, a, b, scale, scale_mode, scale_on_input, out,
                                                                         LayoutU8{0, 0, nullptr, 0});
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_layout_transpose_to_u8(const float* in, int64_t n, int32_t a, int32_t b, const float* scale, int32_t scale_mode,
                               uint8_t* out, void* stream) {
  USF_REQUIRE(in && out && n >= 0 && a > 0 && b > 0, "bad input");
  USF_REQUIRE(scale_mode >= 0 && scale_mode <= 2 && (scale_mode == 0 || scale), "scale_mode 0 (none), 1 (multiply) or 2 (divide)");
  if (n == 0) return USF_OK;
  const long long tiles = (long long)n * ((a + 31) / 32) * ((b + 31) / 32);
  layout_kernel<float, uint8_t><<<ew_grid(tiles * 256, 256), 256, 0, S(stream)>>>(in, n, a, b, scale, scale_mode, 0, out,
                                                                                  LayoutU8{0, 0, nullptr, 0});
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_layout_transpose_u8(const uint8_t* in, int64_t n, int32_t c, int32_t hw, const usf_dequant* dq, const float* scale,
                            int32_t scale_mode, float* out, void* stream) {
  USF_REQUIRE(in && out && n >= 0 && c > 0 && hw > 0, "bad input");
  USF_REQUIRE(dequant_ok(dq), "bad dequantisation (null, or mode not USF_DEQUANT_UNIFORM / USF_DEQUANT_MIDPOINT)");
  USF_REQUIRE(scale_mode >= 0 && scale_mode <= 2 && (scale_mode == 0 || scale), "scale_mode 0 (none), 1 (multiply) or 2 (divide)");
  if (n == 0) return USF_OK;
  const long long tiles = (long long)n * ((c + 31) / 32) * ((hw + 31) / 32);
  layout_kernel<uint8_t><<<ew_grid(tiles * 256, 256), 256, 0, S(stream)>>>(
      in, n, c, hw, scale, scale_mode, 1, out, LayoutU8{dq->seed, dq->row0, reinterpret_cast<const long long*>(dq->dev_params), dq->mode});
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_im2col(const float* in, int64_t ld_in, int64_t n_images, int32_t h, int32_t w, int32_t c, int32_t k, int32_t dilation,
               const float* mask, int32_t relu, const usf_planes* out, int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(in && out && n_images >= 0 && h > 0 && w > 0 && c > 0 && ld_in >= c, "bad input");
  USF_REQUIRE(k >= 1 && (k & 1) && dilation >= 1, "odd kernel size (padding 'same') and dilation >= 1");
  USF_REQUIRE((out->hi == nullptr) == (out->lo == nullptr) && (out->h16 == nullptr) == (out->l16 == nullptr), "planes come as pairs");
  USF_REQUIRE(out->f32 || out->hi || out->bf16 || out->h16, "usf_im2col needs an output plane");
  if (n_images == 0) return USF_OK;
  const OutPlanes o = to_out_planes(out, overflow_flag);
  const long long rows = (long long)n_images * h * w;
  const bool vec = c % 4 == 0 && aligned16(in) && ld_in % 4 == 0 && (!mask || aligned16(mask)) && planes_vec_ok(o);
  if (vec && c % 8 == 0)
    im2col_kernel<8><<<ew_grid(rows * k * k * (c / 8), 256), 256, 0, S(stream)>>>(in, ld_in, rows, h, w, c, k, dilation, mask, relu ? 1 : 0, o);
  else if (vec)
    im2col_kernel<4><<<ew_grid(rows * k * k * (c / 4), 256), 256, 0, S(stream)>>>(in, ld_in, rows, h, w, c, k, dilation, mask, relu ? 1 : 0, o);
  else
    im2col_kernel<1><<<ew_grid(rows * k * k * c, 256), 256, 0, S(stream)>>>(in, ld_in, rows, h, w, c, k, dilation, mask, relu ? 1 : 0, o);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_conv2d_rows(const usf_linear_args* a, const float* act, int64_t ld_act, int64_t n_images, int32_t h, int32_t w,
                    int32_t c_in, int32_t k, int32_t dilation, const float* mask, int32_t relu_in, void* stream) {
  USF_REQUIRE(a && act && a->w && a->w_lo, "null argument (the weight comes as tf32 hi / lo planes)");
  USF_REQUIRE(n_images >= 0 && h > 0 && w > 0 && c_in > 0 && c_in % 16 == 0 && ld_act >= c_in && ld_act % 4 == 0 && aligned16(act),
              "channels-last rows with C % 16 == 0 and 16-byte aligned rows");
  USF_REQUIRE(k >= 1 && (k & 1) && dilation >= 1, "odd kernel size (padding 'same') and dilation >= 1");
  USF_REQUIRE(a->M == n_images * (int64_t)h * w && a->K == k * k * c_in && a->N >= 1, "M = n*h*w, K = k*k*c_in");
  USF_REQUIRE(!mask || aligned16(mask), "unaligned mask");
  USF_REQUIRE(!a->resid && !a->resid_h16 && !a->colscale && !a->postsub, "usf_conv2d_rows: bias / ReLU epilogue only");
  if (a->M == 0) return USF_OK;
  Epilogue ep;
  int rc = make_epilogue(a, &ep);
  if (rc) return rc;
  ConvGeom g{act, ld_act, h, w, c_in, k, dilation, mask, relu_in ? 1 : 0};
  return launch_conv_tc(a, g, ep, S(stream));
}

int usf_pix_encode(const float* x, int64_t ldx, int64_t rows, int32_t c, int32_t hw, const float* mask, int32_t relu,
                   void* out16, int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(x && out16 && rows >= 0 && c > 0 && c <= 32 && hw > 0 && ldx >= c, "bad input (c <= 32 channels)");
  USF_REQUIRE(aligned16(out16), "unaligned pixel planes");
  if (rows == 0) return USF_OK;
  return launch_pix_encode(x, ldx, rows, c, hw, mask, relu ? 1 : 0, out16, overflow_flag, S(stream));
}

int usf_conv2d_pix(const usf_conv_pix_args* a, void* stream) {
  USF_REQUIRE(a != nullptr, "null args");
  USF_REQUIRE(a->a16 && a->w1 && a->bias1 && aligned16(a->a16) && aligned16(a->w1) && aligned16(a->bias1), "null / unaligned operand");
  USF_REQUIRE(a->n_images >= 0 && a->n_images < (1ll << 31) && a->h > 0 && a->w > 0, "bad image extent");
  USF_REQUIRE(a->ksize >= 1 && (a->ksize & 1) && a->dilation >= 1, "odd kernel size (padding 'same') and dilation >= 1");
  USF_REQUIRE(a->n1 >= 4 && a->n1 <= 32 && a->n1 % 4 == 0, "n1: a multiple of 4, at most 32");
  USF_REQUIRE((a->gamma == nullptr) == (a->beta == nullptr), "gamma and beta come as a pair");
  if (a->gated) {
    USF_REQUIRE(a->n1 == 32 && a->w2 && a->bias2 && aligned16(a->w2), "gated block: 32 channels, w2 and bias2");
    USF_REQUIRE(a->out_f32 && a->ld_f32 >= 32 && a->ld_f32 % 4 == 0 && aligned16(a->out_f32), "gated block: fp32 residual stream [rows, 32]");
    USF_REQUIRE(!a->x, "gated block: no coupling update");
  } else {
    USF_REQUIRE(a->out_f32 || a->out16 || a->x, "no output");
    USF_REQUIRE(!a->out_f32 || (a->ld_f32 >= a->n1 && a->ld_f32 % 4 == 0 && aligned16(a->out_f32)), "out_f32: 16-byte aligned rows");
    USF_REQUIRE(!a->x || (a->inv_mask && a->c_x >= 1 && a->c_x <= a->n1 && a->ldx >= a->c_x), "coupling update: x, inv_mask, c_x <= n1");
  }
  USF_REQUIRE(!a->out16 || aligned16(a->out16), "unaligned pixel planes");
  if (a->n_images == 0) return USF_OK;
  return launch_conv_pix(a, S(stream));
}

int usf_masked_add(float* x, int64_t ldx, const float* t, int64_t ldt, int64_t rows, int32_t c, int32_t hw, const float* g,
                   float sign, void* stream) {
  USF_REQUIRE(x && t && g && rows >= 0 && c > 0 && hw > 0 && ldx >= c && ldt >= c, "bad input");
  if (rows == 0) return USF_OK;
  masked_add_kernel<<<ew_grid(rows * c, 256), 256, 0, S(stream)>>>(x, ldx, t, ldt, rows, c, hw, g, sign);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_sub_rows(float* out, const float* v, int64_t n, void* stream) {
  USF_REQUIRE(out && v && n >= 0, "bad input");
  if (n == 0) return USF_OK;
  sub_rows_kernel<<<ew_grid(n, 256), 256, 0, S(stream)>>>(out, v, n);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_leaky_relu(const float* x, int64_t ldx, int64_t rows, int32_t d, float slope, float* y, int64_t ldy,
                   float* neg_count, void* stream) {
  USF_REQUIRE(x && y && d > 0 && rows >= 0, "bad input");
  if (rows == 0) return USF_OK;
  leaky_relu_kernel<<<ew_grid(rows * 32, 256), 256, 0, S(stream)>>>(x, ldx, rows, d, slope, y, ldy, neg_count);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_permute(const float* x, int64_t ldx, int64_t rows, int32_t d, const int32_t* perm, float* y, int64_t ldy,
                void* stream) {
  USF_REQUIRE(x && y && perm && d > 0 && rows >= 0, "bad input");
  USF_REQUIRE(x != y, "permute cannot run in place");
  if (rows == 0) return USF_OK;
  permute_kernel<<<ew_grid(rows * d, 256), 256, 0, S(stream)>>>(x, ldx, rows, d, perm, y, ldy);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_lu_assemble(const float* L_raw, const float* U_raw, int32_t d, int64_t ld_raw, float* L, float* U,
                    int64_t ld_out, int32_t transpose_u, void* stream) {
  USF_REQUIRE(d > 0 && (L || U), "bad input");
  USF_REQUIRE((!L || L_raw) && (!U || U_raw), "missing raw matrix");
  lu_assemble_kernel<<<ew_grid((long long)d * d, 256), 256, 0, S(stream)>>>(L_raw, U_raw, d, ld_raw, L, U, ld_out, transpose_u);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_lu_logabsdet(const float* U_raw, int32_t d, int64_t ld, float* out, void* stream) {
  USF_REQUIRE(U_raw && out && d > 0, "bad input");
  logabs_kernel<<<1, 1024, 0, S(stream)>>>(U_raw, d, ld + 1, out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_vec_logabs(const float* v, int64_t n, float* out, void* stream) {
  USF_REQUIRE(v && out && n > 0, "bad input");
  logabs_kernel<<<1, 1024, 0, S(stream)>>>(v, n, 1, out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int64_t usf_tri_inverse_work_floats(int32_t d) {
  const int64_t nb = (d + TI_NB - 1) / TI_NB;
  return nb * TI_NB * TI_NB + 2LL * d * d;
}

int usf_transpose(const float* in, int32_t rows, int32_t cols, int64_t ld_in, float* out, int64_t ld_out, void* stream) {
  USF_REQUIRE(in && out && rows > 0 && cols > 0 && in != out, "bad input");
  dim3 grid((cols + 31) / 32, (rows + 31) / 32);
  transpose_kernel<<<grid, 256, 0, S(stream)>>>(in, rows, cols, ld_in, out, ld_out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_tri_inverse(const float* T, int32_t d, int64_t ldt, int32_t lower, int32_t unit_diag, float* X, int64_t ldx,
                    float* work, void* stream) {
  USF_REQUIRE(T && X && work && d > 0 && T != X, "bad input");
  const int nb = (d + TI_NB - 1) / TI_NB;
  float* dinv = work;
  if (lower) {
    tri_diag_inverse_kernel<<<nb, TI_NB, 0, S(stream)>>>(T, d, ldt, unit_diag, dinv);
    tri_panel_sweep_kernel<<<nb, 256, 0, S(stream)>>>(T, d, ldt, dinv, X, ldx);
    USF_CUDA_OK(cudaGetLastError());
    return USF_OK;
  }
  float* Tt = work + (int64_t)nb * TI_NB * TI_NB;
  float* Xt = Tt + (int64_t)d * d;
  int rc = usf_transpose(T, d, d, ldt, Tt, d, stream);
  if (rc) return rc;
  tri_diag_inverse_kernel<<<nb, TI_NB, 0, S(stream)>>>(Tt, d, d, unit_diag, dinv);
  tri_panel_sweep_kernel<<<nb, 256, 0, S(stream)>>>(Tt, d, d, dinv, Xt, d);
  USF_CUDA_OK(cudaGetLastError());
  return usf_transpose(Xt, d, d, d, X, ldx, stream);
}

int usf_scale_rows_cols(const float* in, int32_t rows, int32_t cols, int64_t ld_in, const float* rowf,
                        const float* colf, float* out, int64_t ld_out, void* stream) {
  USF_REQUIRE(in && out && rows > 0 && cols > 0, "bad input");
  scale_rows_cols_kernel<<<ew_grid((long long)rows * cols, 256), 256, 0, S(stream)>>>(in, rows, cols, ld_in, rowf, colf, out, ld_out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_split_tf32(const float* in, int64_t rows, int32_t cols, int64_t ld_in, float* hi, float* lo, int64_t ld_out,
                   void* stream) {
  USF_REQUIRE(in && hi && rows > 0 && cols > 0, "bad input");
  split_tf32_kernel<<<ew_grid(rows * cols, 256), 256, 0, S(stream)>>>(in, rows, cols, ld_in, hi, lo, ld_out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_to_bf16(const float* in, int64_t rows, int32_t cols, int64_t ld_in, void* out, int64_t ld_out, void* stream) {
  USF_REQUIRE(in && out && rows > 0 && cols > 0, "bad input");
  to_bf16_kernel<<<ew_grid(rows * cols, 256), 256, 0, S(stream)>>>(in, rows, cols, ld_in, reinterpret_cast<__nv_bfloat16*>(out), ld_out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_split_f16(const float* in, int64_t rows, int32_t cols, int64_t ld_in, void* hi, void* lo, int64_t ld_out,
                  int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(in && hi && lo && rows > 0 && cols > 0, "bad input");
  split_f16_kernel<<<ew_grid(rows * cols, 256), 256, 0, S(stream)>>>(in, rows, cols, ld_in, reinterpret_cast<__half*>(hi),
                                                                     reinterpret_cast<__half*>(lo), ld_out, overflow_flag);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_householder_right(float* W, int32_t d, int64_t ld, const float* v, float* work, void* stream) {
  USF_REQUIRE(W && v && work && d > 0, "bad input");
  householder_matvec_kernel<<<(d + 7) / 8, 256, 0, S(stream)>>>(W, d, ld, v, work);
  householder_rank1_kernel<<<ew_grid((long long)d * d, 256), 256, 0, S(stream)>>>(W, d, ld, v, work);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

static int matmul_f64_launch(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int32_t M,
                             int32_t N, int32_t K, int32_t tri, void* stream) {
  USF_REQUIRE(A && B && C && M > 0 && N > 0 && K > 0, "bad input");
  USF_REQUIRE(C != A && C != B, "matmul_f64 cannot run in place");
  USF_REQUIRE(tri == USF_TRI_NONE || ((tri == USF_TRI_LOWER_UPPER || tri == USF_TRI_UPPER_LOWER) && M == K && N == K),
              "matmul_f64: triangular products are square");
  USF_REQUIRE((M + 63) / 64 <= 65535, "matmul_f64: too many row blocks");
  // fp64 tensor-core tiles: 128 x 128 once they fill the SMs twice over, else 64 x 64 (more CTAs for the 784-wide operators)
  const long long big = (long long)((N + 127) / 128) * ((M + 127) / 128);
  if (big >= 2LL * num_sms())
    matmul_f64_mma_kernel<128, 128, 64, 32><<<dim3((N + 127) / 128, (M + 127) / 128), 256, 0, S(stream)>>>(A, lda, B, ldb, C, ldc, M, N, K, tri);
  else
    matmul_f64_mma_kernel<64, 64, 32, 32><<<dim3((N + 63) / 64, (M + 63) / 64), 128, 0, S(stream)>>>(A, lda, B, ldb, C, ldc, M, N, K, tri);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_matmul_f64(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int32_t M,
                   int32_t N, int32_t K, void* stream) {
  return matmul_f64_launch(A, lda, B, ldb, C, ldc, M, N, K, USF_TRI_NONE, stream);
}

int usf_matmul_f64_tri(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int32_t d,
                       int32_t tri, void* stream) {
  return matmul_f64_launch(A, lda, B, ldb, C, ldc, d, d, d, tri, stream);
}

int usf_plan_create(usf_plan** plan, int32_t d_in, int32_t mode, int64_t max_rows) {
  USF_REQUIRE(plan && d_in > 0 && max_rows > 0 && mode >= USF_MODE_FP32 && mode <= USF_MODE_BF16, "bad input");
  usf_plan* p = new (std::nothrow) usf_plan();
  USF_REQUIRE(p != nullptr, "out of host memory");
  p->d_in = d_in;
  p->mode = mode;
  p->max_rows = max_rows;
  *plan = p;
  return USF_OK;
}

int usf_plan_add_linear(usf_plan* p, const usf_plan_linear* st) {
  USF_REQUIRE(p && st && !p->finalized, "bad input (plan null or already finalized)");
  USF_REQUIRE(st->N > 0 && st->K > 0 && st->w, "bad step");
  USF_REQUIRE(st->src == USF_PLAN_SRC_STREAM || st->src == USF_PLAN_SRC_HIDDEN, "bad step source");
  USF_REQUIRE(st->dst >= USF_PLAN_DST_STREAM && st->dst <= USF_PLAN_DST_SEGMENT, "bad step destination");
  USF_REQUIRE(st->src == USF_PLAN_SRC_STREAM || !p->steps.empty(), "the first step reads the stream");
  p->steps.push_back(*st);
  return USF_OK;
}

int usf_plan_set_base(usf_plan* p, int32_t base_kind, const float* loc, const float* scale, float add_const) {
  USF_REQUIRE(p && loc && scale && (base_kind == USF_BASE_LAPLACE || base_kind == USF_BASE_NORMAL), "bad input");
  p->base_kind = base_kind;
  p->loc = loc;
  p->scale = scale;
  p->add_const = add_const;
  return USF_OK;
}

int64_t usf_plan_workspace_bytes(const usf_plan* p) {
  if (!p) return 0;
  int64_t ws = p->d_in, wh = 8;
  for (const auto& st : p->steps) {
    if (st.dst == USF_PLAN_DST_HIDDEN) wh = st.N > wh ? st.N : wh;
    if (st.dst == USF_PLAN_DST_STREAM) ws = st.N > ws ? st.N : ws;
  }
  // the ingest copy of the input may need the fp32 plane too (unaligned caller tensors in the tf32 / simt modes)
  return 2 * (int64_t)planes_bytes(stream_planes(p->mode) | 1, p->max_rows, ws) +
         2 * (int64_t)planes_bytes(hidden_planes(p->mode), p->max_rows, wh) + (int64_t)p->max_rows * pad_to(ws, 8) * 4 + 256;
}

int usf_plan_finalize(usf_plan* p) {
  USF_REQUIRE(p && !p->finalized && !p->steps.empty(), "bad plan");
  USF_REQUIRE(p->steps.back().dst == USF_PLAN_DST_STREAM, "the last step of a plan writes the stream");
  int64_t ws = p->d_in, wh = 8;
  int32_t width = p->d_in;
  for (const auto& st : p->steps) {
    if (st.dst == USF_PLAN_DST_HIDDEN) wh = st.N > wh ? st.N : wh;
    if (st.dst == USF_PLAN_DST_STREAM) { ws = st.N > ws ? st.N : ws; width = st.N; }
  }
  p->out_width = width;
  const size_t total = (size_t)usf_plan_workspace_bytes(p);
  {   // legal even if the calling thread is capturing a graph (thread-local / global capture modes forbid cudaMalloc)
    RelaxedCaptureMode relaxed;
    USF_CUDA_OK(cudaMalloc(&p->mem, total));
  }
  char* at = reinterpret_cast<char*>(p->mem);
  for (int i = 0; i < 2; ++i) carve_planes(&p->x[i], stream_planes(p->mode) | 1, p->max_rows, ws, at);
  for (int i = 0; i < 2; ++i) carve_planes(&p->h[i], hidden_planes(p->mode), p->max_rows, wh, at);
  p->fin = reinterpret_cast<float*>(at);
  p->ld_fin = pad_to(ws, 8);
  p->finalized = true;
  return USF_OK;
}

int usf_flow_apply(const usf_plan* p, const float* x, int64_t ldx, int64_t rows, float* z, int64_t ldz, int32_t* overflow_flag,
                   void* stream) {
  return plan_run(p, PlanInput{x, nullptr, nullptr}, ldx, rows, z, ldz, overflow_flag, stream);
}

int usf_flow_logprob(const usf_plan* p, const float* x, int64_t ldx, int64_t rows, float* out, int32_t* overflow_flag,
                     void* stream) {
  USF_REQUIRE(p && p->finalized && p->base_kind >= 0 && out, "plan without a base density (usf_plan_set_base)");
  int rc = plan_run(p, PlanInput{x, nullptr, nullptr}, ldx, rows, p->fin, p->ld_fin, overflow_flag, stream);
  if (rc) return rc;
  return usf_base_logprob(p->fin, nullptr, p->ld_fin, rows, p->out_width, p->loc, p->scale, p->base_kind, p->add_const, out,
                          stream);
}

int usf_flow_logprob_u8(const usf_plan* p, const uint8_t* x, int64_t ldx, int64_t rows, const usf_dequant* dq, float* out,
                        int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(p && p->finalized && p->base_kind >= 0 && out, "plan without a base density (usf_plan_set_base)");
  USF_REQUIRE(x && ldx >= p->d_in, "bad input (x null or ldx < d_in)");
  USF_REQUIRE(dequant_ok(dq), "bad dequantisation (null, or mode not USF_DEQUANT_UNIFORM / USF_DEQUANT_MIDPOINT)");
  int rc = plan_run(p, PlanInput{nullptr, x, dq}, ldx, rows, p->fin, p->ld_fin, overflow_flag, stream);
  if (rc) return rc;
  return usf_base_logprob(p->fin, nullptr, p->ld_fin, rows, p->out_width, p->loc, p->scale, p->base_kind, p->add_const, out,
                          stream);
}

int usf_plan_destroy(usf_plan* p) {
  if (!p) return USF_OK;
  if (p->mem) {
    // a host may destroy a plan from a finaliser that runs while this thread captures a graph: cudaFree would invalidate
    // the capture in the thread-local / global modes
    RelaxedCaptureMode relaxed;
    cudaFree(p->mem);
  }
  delete p;
  return USF_OK;
}

int usf_planes_glue(const usf_glue_args* g, void* stream) {
  USF_REQUIRE(g != nullptr, "null args");
  GlueArgs a;
  a.h = reinterpret_cast<const __half*>(g->h);
  a.l = reinterpret_cast<const __half*>(g->l);
  a.ld = g->ld;
  a.src_f32 = g->src_f32;
  a.ld_src = g->ld_src;
  a.rows = g->rows;
  a.n = g->n;
  a.mask_h = reinterpret_cast<const __half*>(g->mask_h);
  a.ld_mask = g->ld_mask;
  a.sign = g->sign;
  a.out_h = reinterpret_cast<__half*>(g->out_h);
  a.out_l = reinterpret_cast<__half*>(g->out_l);
  a.ld_out = g->ld_out;
  a.t_h = reinterpret_cast<__half*>(g->t_h);
  a.t_l = reinterpret_cast<__half*>(g->t_l);
  a.ld_t = g->ld_t;
  a.colsum = g->colsum;
  a.mul = g->mul;
  a.ld_mul = g->ld_mul;
  a.colsum2 = g->colsum2;
  a.overflow_flag = g->overflow_flag;
  USF_REQUIRE(a.rows >= 0 && a.n >= 0, "negative extent");
  USF_REQUIRE((a.h == nullptr) == (a.l == nullptr) && (a.out_h == nullptr) == (a.out_l == nullptr) &&
                  (a.t_h == nullptr) == (a.t_l == nullptr), "planes come as (hi, lo) pairs");
  USF_REQUIRE(a.rows < (1LL << 31) && (a.rows + GL_TILE - 1) / GL_TILE <= 65535, "planes glue: too many rows for one launch");
  return launch_planes_glue(a, S(stream));
}

int usf_base_backward(const float* z, int64_t ldz, int64_t rows, int32_t d, const float* loc, const float* scale,
                      int32_t kind, void* g_h, void* g_l, int64_t ld_g, void* t_h, void* t_l, int64_t ld_t, float* dloc,
                      float* dscale, void* stream) {
  USF_REQUIRE(z && loc && scale && g_h && g_l && rows >= 0 && d > 0 && d % 8 == 0, "bad input");
  USF_REQUIRE(kind == USF_BASE_LAPLACE || kind == USF_BASE_NORMAL, "unknown base kind");
  USF_REQUIRE((t_h == nullptr) == (t_l == nullptr), "planes come as (hi, lo) pairs");
  USF_REQUIRE(aligned16(g_h) && aligned16(g_l) && ld_g % 8 == 0 && (!t_h || (aligned16(t_h) && aligned16(t_l) && ld_t % 8 == 0)),
              "base backward: 16-byte aligned planes");
  if (rows == 0) return USF_OK;
  USF_REQUIRE((rows + GL_TILE - 1) / GL_TILE <= 65535, "base backward: too many rows for one launch");
  dim3 grid((d + GL_TILE - 1) / GL_TILE, (unsigned)((rows + GL_TILE - 1) / GL_TILE));
  base_backward_kernel<<<grid, 256, 0, S(stream)>>>(z, ldz, rows, d, loc, scale, kind, reinterpret_cast<__half*>(g_h),
                                                    reinterpret_cast<__half*>(g_l), ld_g, reinterpret_cast<__half*>(t_h),
                                                    reinterpret_cast<__half*>(t_l), ld_t, dloc, dscale);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_mat_prep(const float* src, int64_t ld_src, int32_t rows, int32_t cols, int32_t transpose, const int32_t* row_idx,
                 const int32_t* col_idx, float scale, float* out_f32, int64_t ld_f32, void* out_h, void* out_l, int64_t ld_16,
                 void* outT_h, void* outT_l, int64_t ld_T, int32_t* overflow_flag, void* stream) {
  USF_REQUIRE(src && rows > 0 && cols > 0 && (out_f32 || out_h || outT_h), "bad input");
  USF_REQUIRE((out_h == nullptr) == (out_l == nullptr) && (outT_h == nullptr) == (outT_l == nullptr),
              "planes come as (hi, lo) pairs");
  USF_REQUIRE(src != out_f32, "mat_prep cannot run in place");
  mat_prep_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), 256, 0, S(stream)>>>(
      src, ld_src, rows, cols, transpose, row_idx, col_idx, scale, out_f32, ld_f32, reinterpret_cast<__half*>(out_h),
      reinterpret_cast<__half*>(out_l), ld_16, reinterpret_cast<__half*>(outT_h), reinterpret_cast<__half*>(outT_l), ld_T,
      overflow_flag);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_rowdot(const float* W, int64_t ld, int32_t n_rows, int32_t K, const int32_t* row_idx, const float* v, float alpha,
               float* out, void* stream) {
  USF_REQUIRE(W && v && out && n_rows > 0 && K > 0, "bad input");
  rowdot_kernel<<<(n_rows * 32 + 255) / 256, 256, 0, S(stream)>>>(W, ld, n_rows, K, row_idx, v, alpha, out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_colcomb(const float* W, int64_t ld, int32_t rows, int32_t cols, const float* v, float alpha, float* out, void* stream) {
  USF_REQUIRE(W && v && out && rows > 0 && cols > 0, "bad input");
  colcomb_kernel<<<dim3((cols + 255) / 256, (rows + CC_ROWS - 1) / CC_ROWS), 256, 0, S(stream)>>>(W, ld, rows, cols, v, alpha, out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_rank1(float* A, int64_t ld, int32_t rows, int32_t cols, const float* u, const float* v, float alpha, void* stream) {
  USF_REQUIRE(A && u && v && rows > 0 && cols > 0, "bad input");
  rank1_kernel<<<ew_grid((long long)rows * cols, 256), 256, 0, S(stream)>>>(A, ld, rows, cols, u, v, alpha);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_tri_mask(const float* src, int64_t ld_src, int32_t d, int32_t mode, float scale, const float* diag_src,
                 int64_t ld_diag, float coef, float* out, int64_t ld_out, void* stream) {
  USF_REQUIRE(src && out && d > 0 && (mode == 0 || mode == 1), "bad input");
  tri_mask_kernel<<<ew_grid((long long)d * d, 256), 256, 0, S(stream)>>>(src, ld_src, d, mode, scale, diag_src, ld_diag, coef,
                                                                         out, ld_out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int usf_tri_inverse_batched(const float* T, float* X, float* tmp, int32_t d, int64_t ld, int64_t mat_stride, int32_t n_mats,
                            uint32_t unit_mask, void* stream) {
  return launch_tri_inverse_batched(T, X, tmp, d, ld, mat_stride, n_mats, unit_mask, S(stream));
}

int usf_softplus(const float* in, int64_t n, float* out, void* stream) {
  USF_REQUIRE(in && out && n > 0, "bad input");
  softplus_kernel<<<ew_grid(n, 256), 256, 0, S(stream)>>>(in, n, out);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

}  // extern "C"
