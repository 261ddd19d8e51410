// Internal launch interface shared by plan.cu and the kernel files.
#pragma once
#include "common.cuh"

namespace acr {

struct TensorRef {         // resolved acr_b200_tensor: absolute base pointer, per-image extents
  void* ptr;
  int C, H, W, pix_stride, dtype;
  __host__ __device__ size_t img_stride() const { return (size_t)H * W * pix_stride; }
};

struct ConvArgs {
  TensorRef in, out, res;
  const void* w;           // [cout_pad][k*k][cin_pad] 16-bit
  const float* bias;       // [cout_pad] (or [B][cout_pad] when bias_per_image)
  int k, stride, relu, has_res, cin_pad, cout_pad, bias_per_image, pow11_ch0, batch;
  int xpair;               // weights are the x-paired expansion of a 32->32 conv (ACR_CONV_XPAIR): side taps are 32x32 corners
  TensorRef ext[3];        // ACR_CONV_EXTRA: up to three more terms added before the activation (HRNet fuse sums folded into
  int n_ext, ext_shift[3]; // the producing conv): term e is read at pixel (oy >> shift, ox >> shift) = nearest upsampling
  int s2x;                 // ACR_CONV_S2X: 3x3 stride-2 conv of a dense 32-channel tensor given as its x-paired view (H, W/2, 64)
};

struct FuseArgs {
  TensorRef out, in[4];
  int n_in, shift[4], relu, batch;
};

// every launcher returns an ACR_B200_* status and performs exactly ONE kernel launch
int launch_stem(const TensorRef& img, const TensorRef& out, const float* w, const float* bias, int batch,
                int act_dtype, cudaStream_t st);
int launch_im2col_stem(const TensorRef& img, const TensorRef& out, int batch, int act_dtype, cudaStream_t st);
// stem conv on the tensor cores with the A operand built in shared memory from the uint8 frame (stem_tc.cu): w = packed
// [64][32] 16-bit (tap-major K, BN folded), bias fp32 [64]
// conv_tc.cu: tensor map (128 bytes, 64-byte aligned) for TMA stores of [4 rows][8 px][64 ch] slabs into an NHWC tensor
int encode_slab_store_map(void* tmap, const TensorRef& out, int channels, int batch, int act_dtype);
int launch_stem_tc(const TensorRef& img, const TensorRef& out, const void* w, const float* bias, int batch, int act_dtype,
                   cudaStream_t st);
int launch_conv_ref(const ConvArgs& a, int act_dtype, cudaStream_t st);
int launch_fuse(const FuseArgs& a, int act_dtype, cudaStream_t st);
int launch_bilinear2x(const TensorRef& in, const TensorRef& out, int batch, int act_dtype, cudaStream_t st);
int launch_coord(const TensorRef& out, int c_off, int batch, int act_dtype, cudaStream_t st);
// attention pooling, split-softmax partials: part (B, NCHUNK, 256*32 + 64) fp32
constexpr int POOL_CHUNKS = 16;
constexpr int POOL_PART_FLOATS = 256 * 32 + 64;
int launch_pool(const TensorRef& feat, const TensorRef& logits, float* part, int batch, int act_dtype,
                cudaStream_t st);
// pool_tc.cu: the same contraction on tcgen05 / TMEM fed by TMA; launch_pool uses it for the shapes it takes
bool pool_tc_enabled();
bool pool_tc_takes(const TensorRef& feat, const TensorRef& logits);
int launch_pool_tc(const TensorRef& feat, const TensorRef& logits, float* part, int batch, int act_dtype, cudaStream_t st);
struct PartHeadArgs {
  const float* part;           // pool partials
  float* pooled;               // (B,256,32) fp32 normalised attention-pooled features (output)
  const float* lc_w[2];        // LocallyConnected2d weights (6,256,16) for l, r
  const float* shape_w;        // cam_shape_layers[1] 1x1 conv (64,256) fp32
  const float* shape_b;        // (64)
  const float* lin_w[2];       // Linear (10,1024)
  const float* lin_b[2];       // (10)
  const float* fin_w[2];       // contact_layers[4|5] (109,218) fp32
  const float* fin_b[2];       // (109)
  float* bias_img[2];          // (B,112) per-image bias of the folded 1x1 conv (output)
  float* pare[2];              // (B,106) contact offsets (96) + shape offsets (10) (output)
  int batch;
};
int launch_parthead(const PartHeadArgs& a, cudaStream_t st);
// fp32-storage validation plan (validate_f32.cu): same ops, fp32 tensors, fp64 accumulation
int launch_stem_f32(const TensorRef& img, const TensorRef& out, const float* w, const float* bias, int batch, cudaStream_t st);
int launch_conv_f32(const ConvArgs& a, cudaStream_t st);
int launch_fuse_f32(const FuseArgs& a, cudaStream_t st);
int launch_bilinear2x_f32(const TensorRef& in, const TensorRef& out, int batch, cudaStream_t st);
int launch_coord_f32(const TensorRef& out, int c_off, int batch, cudaStream_t st);
int launch_pool_f32(const TensorRef& feat, const TensorRef& logits, float* part, int batch, cudaStream_t st);
// tcgen05 implicit-GEMM conv (conv_tc.cu)
struct ConvTcPlan;   // holds the TMA tensor maps of one conv op
int conv_tc_prepare(const ConvArgs& a, int act_dtype, ConvTcPlan** out);
int conv_tc_launch(const ConvTcPlan* p, cudaStream_t st);
// the plan's kernel instance and schedule as the ACR_CONV_INFO_* fields of include/acr_b200.h (first n_info of them)
int conv_tc_describe(const ConvTcPlan* p, int32_t* info, int n_info);
void conv_tc_free(ConvTcPlan* p);

}  // namespace acr
