// Whole-stack entry points (SURVEY 8b: usf_plan_create / usf_flow_logprob / usf_plan_destroy): the launch sequence of one
// direction of a layer stack -- ingest, the contractions with their fused epilogues, the base density -- owned by the
// library, so that a host that is not Python (or a small batch, where ~25 Python -> ctypes calls cost more than the
// kernels) makes ONE call per batch.  The plan mirrors engine.Program._run_chunk for programs made of contractions only
// (every USFlow with DenseNN conditioners: reference flows.py:225-245 for the density direction, :45-55 for sampling).
#pragma once
#include <vector>

#include "common.cuh"

struct usf_plan {
  int32_t d_in = 0, mode = 0;
  int64_t max_rows = 0;
  std::vector<usf_plan_linear> steps;
  bool finalized = false;
  int32_t base_kind = -1;
  const float* loc = nullptr;
  const float* scale = nullptr;
  float add_const = 0.f;
  int32_t out_width = 0;
  // workspaces (device): two stream buffers, two hidden buffers, the fp32 result
  void* mem = nullptr;
  usf_planes x[2], h[2];
  float* fin = nullptr;
  int64_t ld_fin = 0;
};

namespace usf {

inline int64_t pad_to(int64_t n, int64_t m) { return (n + m - 1) / m * m; }

// which planes an activation of a mode carries: bit 0 f32, 1 hi/lo, 2 bf16, 3 h16/l16
inline int stream_planes(int mode) {
  switch (mode) {
    case USF_MODE_FP32: return 8;
    case USF_MODE_FP32_TF32: return 2;
    case USF_MODE_BF16: return 4 | 1;
    default: return 1;      // tf32 / simt
  }
}
inline int hidden_planes(int mode) { return mode == USF_MODE_BF16 ? 4 : stream_planes(mode); }
inline int operand_planes(int mode) { return hidden_planes(mode); }

inline size_t planes_bytes(int set, int64_t rows, int64_t width) {
  const int64_t ld = pad_to(width, 8);
  size_t b = 0;
  if (set & 1) b += (size_t)rows * ld * 4;
  if (set & 2) b += (size_t)rows * ld * 8;
  if (set & 4) b += (size_t)rows * ld * 2;
  if (set & 8) b += (size_t)rows * ld * 4;
  return (b + 255) / 256 * 256;
}
inline void carve_planes(usf_planes* p, int set, int64_t rows, int64_t width, char*& at) {
  const int64_t ld = pad_to(width, 8);
  memset(p, 0, sizeof(*p));
  char* start = at;
  if (set & 1) { p->f32 = reinterpret_cast<float*>(at); p->ld_f32 = ld; at += (size_t)rows * ld * 4; }
  if (set & 2) {
    p->hi = reinterpret_cast<float*>(at); at += (size_t)rows * ld * 4;
    p->lo = reinterpret_cast<float*>(at); at += (size_t)rows * ld * 4;
    p->ld_split = ld;
  }
  if (set & 4) { p->bf16 = at; p->ld_bf16 = ld; at += (size_t)rows * ld * 2; }
  if (set & 8) {
    p->h16 = at; at += (size_t)rows * ld * 2;
    p->l16 = at; at += (size_t)rows * ld * 2;
    p->ld_16 = ld;
  }
  at = start + planes_bytes(set, rows, width);
}
// view of the columns [c0, ...) of every plane
inline usf_planes seg_planes(const usf_planes& a, int c0) {
  usf_planes v = a;
  if (v.f32) v.f32 += c0;
  if (v.hi) { v.hi += c0; v.lo += c0; }
  if (v.bf16) v.bf16 = reinterpret_cast<char*>(v.bf16) + (size_t)c0 * 2;
  if (v.h16) { v.h16 = reinterpret_cast<char*>(v.h16) + (size_t)c0 * 2; v.l16 = reinterpret_cast<char*>(v.l16) + (size_t)c0 * 2; }
  return v;
}
inline bool has_planes(const usf_planes& a, int set) {
  return (!(set & 1) || a.f32) && (!(set & 2) || a.hi) && (!(set & 4) || a.bf16) && (!(set & 8) || a.h16);
}

// usf_linear arguments from plane sets (the same choices as usflows_b200/ops.py:linear)
inline void fill_linear(usf_linear_args* g, int engine, const usf_planes& a, const usf_plan_linear& st, const usf_planes* resid,
                        const usf_planes& out, int64_t rows, int32_t* flag) {
  memset(g, 0, sizeof(*g));
  g->M = rows; g->N = st.N; g->K = st.K; g->engine = engine;
  if (engine == USF_ENGINE_TC_3XF16) { g->a = a.h16; g->a_lo = a.l16; g->lda = a.ld_16; }
  else if (engine == USF_ENGINE_TC_BF16) { g->a = a.bf16; g->lda = a.ld_bf16; }
  else if (engine == USF_ENGINE_TC_3XTF32) { g->a = a.hi; g->a_lo = a.lo; g->lda = a.ld_split; }
  else if (a.f32) { g->a = a.f32; g->lda = a.ld_f32; }
  else { g->a = a.hi; g->a_lo = engine == USF_ENGINE_SIMT ? a.lo : nullptr; g->lda = a.ld_split; }
  g->w = st.w; g->w_lo = st.w_lo; g->ldw = st.ldw;
  g->bias = st.bias; g->relu = st.relu; g->resid_sign = st.resid_sign;
  if (resid) {
    if (!resid->f32 && !resid->hi && resid->h16) { g->resid_h16 = resid->h16; g->resid_l16 = resid->l16; g->ldr_16 = resid->ld_16; }
    else if (resid->f32) { g->resid = resid->f32; g->ldr = resid->ld_f32; }
    else { g->resid = resid->hi; g->resid_lo = resid->lo; g->ldr = resid->ld_split; }
  }
  if (out.f32) { g->out_f32 = out.f32; g->ld_f32 = out.ld_f32; }
  if (out.hi) { g->out_hi = out.hi; g->out_lo = out.lo; g->ld_split = out.ld_split; }
  if (out.bf16) { g->out_bf16 = out.bf16; g->ld_bf16 = out.ld_bf16; }
  if (out.h16) { g->out_h16 = out.h16; g->out_l16 = out.l16; g->ld_16 = out.ld_16; g->overflow_flag = flag; }
}

inline int plan_ingest(const float* x, int64_t ldx, int64_t rows, int32_t d, const usf_planes& o, int32_t* flag, void* stream) {
  if (o.h16) return usf_ingest_f16(x, ldx, rows, d, nullptr, nullptr, nullptr, o.h16, o.l16, o.ld_16, flag, stream);
  return usf_ingest(x, ldx, rows, d, nullptr, nullptr, nullptr, o.f32, o.ld_f32, o.hi, o.lo, o.ld_split, o.bf16, o.ld_bf16, stream);
}

// the caller's rows: fp32, or 8-bit values with their dequantisation (then step 0 always ingests: no fp32 tensor to read)
struct PlanInput {
  const float* f32;
  const uint8_t* u8;
  const usf_dequant* dq;
};

// runs the contraction chain; the last step writes fp32 into (z_out, ldz)
inline int plan_run(const usf_plan* p, PlanInput in, int64_t ldx, int64_t rows, float* z_out, int64_t ldz, int32_t* flag,
                    void* stream) {
  USF_REQUIRE(p && p->finalized, "plan not finalized");
  USF_REQUIRE((in.f32 || in.u8) && z_out && rows >= 0 && rows <= p->max_rows, "bad input (rows must not exceed the plan's max_rows)");
  if (rows == 0) return USF_OK;
  const int mode = p->mode;
  const float* x = in.f32;
  usf_planes src;
  memset(&src, 0, sizeof(src));
  src.f32 = const_cast<float*>(x);           // NULL for 8-bit rows: no plane satisfies a consumer, so they are ingested
  src.ld_f32 = ldx;
  usf_planes cur = src, hid;
  memset(&hid, 0, sizeof(hid));
  bool cur_is_src = true;
  int xf = 0, hf = 0;
  int cur_width = p->d_in;
  for (size_t i = 0; i < p->steps.size(); ++i) {
    const usf_plan_linear& st = p->steps[i];
    const bool last = i + 1 == p->steps.size();
    usf_planes a;
    if (st.src == USF_PLAN_SRC_STREAM) {
      const bool in_coupling = st.dst == USF_PLAN_DST_HIDDEN || st.dst == USF_PLAN_DST_SEGMENT;
      const int need = in_coupling ? stream_planes(mode) : operand_planes(mode);
      const bool direct_ok = st.engine == USF_ENGINE_SIMT || (aligned16(x) && ldx % 4 == 0);
      if (!has_planes(cur, need) || (cur_is_src && !direct_ok)) {
        USF_REQUIRE(cur.f32 != nullptr || (cur_is_src && in.u8), "internal: activation has no fp32 plane to re-encode from");
        xf ^= 1;
        usf_planes b = p->x[xf];
        // only the planes this consumer needs
        if (!(need & 1)) { b.f32 = nullptr; }
        if (!(need & 2)) { b.hi = b.lo = nullptr; }
        if (!(need & 4)) { b.bf16 = nullptr; }
        if (!(need & 8)) { b.h16 = b.l16 = nullptr; }
        int rc = cur_is_src && in.u8 ? usf_ingest_u8(in.u8, ldx, rows, cur_width, in.dq, nullptr, nullptr, nullptr, &b, flag, stream)
                                     : plan_ingest(cur.f32, cur.ld_f32, rows, cur_width, b, flag, stream);
        if (rc) return rc;
        cur = b;
        cur_is_src = false;
      }
      a = st.in_width > 0 ? seg_planes(cur, st.in_col0) : cur;
    } else {
      a = hid;
    }
    usf_planes out;
    memset(&out, 0, sizeof(out));
    const usf_planes* resid = nullptr;
    usf_planes seg;
    usf_linear_args g;
    if (st.dst == USF_PLAN_DST_HIDDEN) {
      hf ^= 1;
      out = p->h[hf];
      if (!(hidden_planes(mode) & 1)) out.f32 = nullptr;
    } else if (st.dst == USF_PLAN_DST_SEGMENT) {       // coupling output, in place on a column segment of the stream
      USF_REQUIRE(!last, "a coupling cannot be the final step of a plan");
      USF_REQUIRE(!cur_is_src, "internal: in-place update of the caller's tensor");
      seg = seg_planes(cur, st.out_col0);
      out = seg;
      resid = &seg;
    } else if (last) {
      out.f32 = z_out;
      out.ld_f32 = ldz;
    } else {
      xf ^= 1;
      out = p->x[xf];
      const int set = stream_planes(mode);
      if (!(set & 1)) out.f32 = nullptr;
    }
    fill_linear(&g, st.engine, a, st, resid, out, rows, flag);
    int rc = usf_linear(&g, stream);
    if (rc) return rc;
    if (st.dst == USF_PLAN_DST_HIDDEN) hid = out;
    else if (st.dst == USF_PLAN_DST_STREAM) { cur = out; cur_is_src = false; cur_width = st.N; }
  }
  return USF_OK;
}

}  // namespace usf
