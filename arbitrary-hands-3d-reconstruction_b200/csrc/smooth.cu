// Temporal smoothing of the MANO parameters between parse and MANO (SURVEY.md 8f-3).
// Replaces (reference, /root/reference): OneEuroFilter / LowPassFilter acr/utils.py:1485-1527,
// smooth_results :1478-1482, smooth_global_rot_matrix :1466-1470 and the per-frame host loop of
// acr/main.py:69-83 (one python filter object per hand type, tensors filtered element-wise on the host
// side of the stream).  Here: one launch, state in a device buffer, no host round trip.
//   filtered quantities per hand: hand pose (45, axis-angle), betas (10), root rotation MATRIX (9,
//   Rodrigues of pose[:3]; the smoothed matrix goes back through rotation_matrix_to_angle_axis).
//   x_hat = lowpass(x, alpha(mincutoff + beta*|lowpass(dx, alpha(dcutoff))|)),  dx = (x - x_prev)*freq,
//   alpha(c) = 1 / (1 + (1/(2 pi c)) / (1/freq)),  freq = 30, beta = 0.7, dcutoff = 1,
//   mincutoff = smooth_coeff (pose, root rotation) | 0.6 (betas).
// Many streams: the state is one block of two banks per stream; a row's bank is (stream_ids[batch_ids[row]],
// hand type).  Without stream ids there is one stream and the bank is the hand type alone.
#include "common.cuh"
#include "rotation.cuh"

namespace acr {

constexpr int SM_ELEMS = 64;            // 45 pose + 10 betas + 9 rotation entries
constexpr int SM_STATE = 4 * SM_ELEMS;  // per hand type: prev_raw, prev_filtered, prev_filtered_dx, [0] = initialised

__device__ __forceinline__ float one_euro_alpha(float cutoff) {
  const float te = 1.0f / 30.0f;
  const float tau = 1.0f / (2.0f * 3.14159265358979323846f * cutoff);
  return 1.0f / (1.0f + tau / te);
}

__global__ void __launch_bounds__(SM_ELEMS) one_euro_kernel(float* __restrict__ poses, float* __restrict__ betas,
                                                            const int32_t* __restrict__ hand_type,
                                                            const float* __restrict__ detection_flag,
                                                            const int64_t* __restrict__ batch_ids,
                                                            const int32_t* __restrict__ stream_ids, int n_streams,
                                                            const int32_t* __restrict__ n_dev, int n_max,
                                                            float* __restrict__ state, float smooth_coeff) {
  __shared__ float s_R[9];
  const int row = blockIdx.x, e = threadIdx.x;
  const int n = n_dev ? min(*n_dev, n_max) : n_max;
  if (row >= n) return;
  if (detection_flag && !(detection_flag[row] > 0.f)) return;   // undetected hands are not filtered (main.py:72-79)
  int bank = hand_type ? (hand_type[row] != 0) : row;
  if (stream_ids) {
    const int s = stream_ids[batch_ids[row]];
    if (s < 0 || s >= n_streams) return;                        // padding slot: no stream, no state touched
    bank += 2 * s;
  }
  float* st = state + (size_t)bank * SM_STATE;
  float* p = poses + (size_t)row * 48;
  float x, mincut;
  if (e < 45) { x = p[3 + e]; mincut = smooth_coeff; }
  else if (e < 55) { x = betas[(size_t)row * 10 + (e - 45)]; mincut = 0.6f; }
  else { float R[9]; rodrigues(p[0], p[1], p[2], R); x = R[e - 55]; mincut = smooth_coeff; }
  const bool init = st[3 * SM_ELEMS] != 0.f;
  float xh, edx;
  if (!init) { xh = x; edx = 0.f; }
  else {
    const float dx = (x - st[e]) * 30.0f;
    const float ad = one_euro_alpha(1.0f);
    edx = ad * dx + (1.0f - ad) * st[2 * SM_ELEMS + e];
    const float a = one_euro_alpha(mincut + 0.7f * fabsf(edx));
    xh = a * x + (1.0f - a) * st[SM_ELEMS + e];
  }
  __syncthreads();   // every thread has read the init flag and its old state
  st[e] = x; st[SM_ELEMS + e] = xh; st[2 * SM_ELEMS + e] = edx;
  if (e == 0) st[3 * SM_ELEMS] = 1.f;
  if (e < 45) p[3 + e] = xh;
  else if (e < 55) betas[(size_t)row * 10 + (e - 45)] = xh;
  else s_R[e - 55] = xh;
  __syncthreads();
  if (e == 0) {
    float aa[3];
    rotmat_to_aa(s_R, aa);
    p[0] = aa[0]; p[1] = aa[1]; p[2] = aa[2];
  }
}

}  // namespace acr

using namespace acr;

extern "C" size_t acr_b200_one_euro_state_floats(void) { return 2 * SM_STATE; }

extern "C" int acr_b200_one_euro_smooth(float* poses, float* betas, const int32_t* hand_type,
                                        const float* detection_flag, const int32_t* n_dev, int n_max,
                                        float* state, float smooth_coeff, void* stream) {
  ACR_CHECK_ARG(n_max >= 0 && (n_max == 0 || (poses && betas && state)), "one_euro_smooth: bad arguments");
  ACR_CHECK_ARG(smooth_coeff > 0.f, "one_euro_smooth: smooth_coeff must be positive");
  if (n_max == 0) return ACR_B200_OK;
  one_euro_kernel<<<n_max, SM_ELEMS, 0, (cudaStream_t)stream>>>(poses, betas, hand_type, detection_flag, nullptr,
                                                                nullptr, 0, n_dev, n_max, state, smooth_coeff);
  ACR_CHECK_LAUNCH();
  return ACR_B200_OK;
}

extern "C" int acr_b200_one_euro_smooth_streams(float* poses, float* betas, const int32_t* hand_type,
                                                const float* detection_flag, const int64_t* batch_ids,
                                                const int32_t* stream_ids, int n_streams, const int32_t* n_dev,
                                                int n_max, float* state, float smooth_coeff, void* stream) {
  ACR_CHECK_ARG(n_max >= 0 && n_streams > 0 && (n_max == 0 || (poses && betas && state)),
                "one_euro_smooth_streams: bad arguments");
  ACR_CHECK_ARG(n_max == 0 || (hand_type && batch_ids && stream_ids),
                "one_euro_smooth_streams: hand_type, batch_ids and stream_ids are required");
  ACR_CHECK_ARG(smooth_coeff > 0.f, "one_euro_smooth_streams: smooth_coeff must be positive");
  if (n_max == 0) return ACR_B200_OK;
  one_euro_kernel<<<n_max, SM_ELEMS, 0, (cudaStream_t)stream>>>(poses, betas, hand_type, detection_flag, batch_ids,
                                                                stream_ids, n_streams, n_dev, n_max, state,
                                                                smooth_coeff);
  ACR_CHECK_LAUNCH();
  return ACR_B200_OK;
}
