// usf_conv2d_pix / usf_pix_encode launchers (own translation unit: parallel build).
#include "conv_pix.cuh"

namespace usf {

// taps per TMEM accumulation chain: 3 (96 K-elements) in the gated block, 2 (the flat engine's chain length) in a plain
// convolution (measured on a B200, DESIGN.md 4.3)
constexpr int PIX_CHAIN_TAPS_GATED = 3, PIX_CHAIN_TAPS_PLAIN = 2;
// gated block: chains of the next tile issued in front of a tile's 1 x 1 gate contraction
constexpr int PIX_GATE_AT = 1;

static int make_pix_map(CUtensorMap* map, const void* ptr, long long n_images, int H, int W, int hr, int imgs) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return fail(USF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available%s%s");
  cuuint64_t dims[4] = {64, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n_images};
  cuuint64_t strides[3] = {(cuuint64_t)convpix::PIX_BYTES, (cuuint64_t)W * convpix::PIX_BYTES,
                           (cuuint64_t)H * W * convpix::PIX_BYTES};
  cuuint32_t box[4] = {64, (cuuint32_t)W, (cuuint32_t)hr, (cuuint32_t)imgs};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof(g_err), "cuTensorMapEncodeTiled (pixel planes) failed with CUresult %d (n=%lld h=%d w=%d box %d x %d)",
             (int)r, n_images, H, W, hr, imgs);
    return USF_ERR_CUDA;
  }
  return USF_OK;
}

int launch_conv_pix(const usf_conv_pix_args* a, cudaStream_t st) {
  PixArgs p;
  memset(&p, 0, sizeof(p));
  int imgs, hr, tpi;
  if (!conv_pix_geometry(a->h, a->w, &imgs, &hr, &tpi))
    return fail(USF_ERR_UNSUPPORTED, "usf_conv2d_pix: image rows wider than 256 pixels%s%s");
  if (imgs > a->n_images) imgs = (int)a->n_images;       // (a box never exceeds the tensor: small batches)
  const int taps = a->ksize * a->ksize;
  const int stages = conv_pix_stages(taps, a->gated);
  if (stages == 0) return fail(USF_ERR_UNSUPPORTED, "usf_conv2d_pix: the weight leaves no room for the pipeline in shared memory%s%s");
  p.n_images = (int)a->n_images; p.H = a->h; p.W = a->w; p.HW = a->h * a->w;
  p.rows = a->n_images * (long long)p.HW;
  p.ksize = a->ksize; p.dil = a->dilation; p.taps = taps;
  p.imgs = imgs; p.hr = hr; p.tiles_per_img = tpi;
  p.n_tiles = tpi == 1 ? (a->n_images + imgs - 1) / imgs : a->n_images * (long long)tpi;
  p.stages = stages;
  p.chain_taps = a->gated ? PIX_CHAIN_TAPS_GATED : PIX_CHAIN_TAPS_PLAIN;
  if (p.chain_taps > stages - 1) p.chain_taps = stages - 1;   // a chain holds its stages until its last product is issued
  if (p.chain_taps > taps) p.chain_taps = taps;
  p.gate_at = PIX_GATE_AT;
  p.box_bytes = (unsigned)(convpix::PIX_BYTES * a->w * hr * imgs);
  p.gated = a->gated ? 1 : 0;
  p.bias1 = a->bias1; p.n1 = a->n1; p.relu1 = a->relu1;
  p.gamma = a->gamma; p.beta = a->beta; p.eps = a->eps;
  p.out_f32 = a->out_f32; p.ld_f32 = a->ld_f32;
  p.out16 = reinterpret_cast<__half*>(a->out16); p.relu_planes = a->relu_planes;
  p.x = a->x; p.ldx = a->ldx; p.inv_mask = a->inv_mask; p.sign = a->sign; p.c_x = a->c_x;
  p.bias2 = a->bias2; p.post_relu = a->post_relu;
  p.overflow_flag = a->overflow_flag;

  auto kern = convpix::conv_pix_kernel;
  const size_t smem = conv_pix_smem_bytes(taps, p.gated);
  static size_t attr_bytes_dev[MAX_DEVICES] = {0};
  size_t& attr_bytes = attr_bytes_dev[current_device_slot()];
  if (smem > attr_bytes) {
    USF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_bytes = smem;
  }
  CUtensorMap ma, mw1, mw2;
  int rc;
  if ((rc = make_pix_map(&ma, a->a16, a->n_images, a->h, a->w, hr, imgs))) return rc;
  if ((rc = make_operand_map(&mw1, a->w1, 32, (long long)taps * 64, (long long)taps * 64, 32, 2))) return rc;
  if (p.gated) {
    if ((rc = make_operand_map(&mw2, a->w2, 64, 64, 64, 64, 2))) return rc;
  } else {
    mw2 = mw1;
  }
  const int grid = (int)(p.n_tiles < num_sms() ? p.n_tiles : num_sms());
  USF_CUDA_OK(launch_chain(kern, dim3(grid), dim3(convpix::PIX_THREADS), smem, st, ma, mw1, mw2, p));
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

int launch_pix_encode(const float* x, long long ldx, long long rows, int c, int hw, const float* mask, int relu, void* out16,
                      int* overflow_flag, cudaStream_t st) {
  const long long n = rows * 4;
  convpix::pix_encode_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, ldx, rows, c, hw, mask, relu,
                                                                         reinterpret_cast<__half*>(out16), overflow_flag);
  USF_CUDA_OK(cudaGetLastError());
  return USF_OK;
}

}  // namespace usf
