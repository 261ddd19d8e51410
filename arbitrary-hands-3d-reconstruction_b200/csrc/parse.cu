// Centre parsing + parameter sampling + 6D->axis-angle, without a single host sync.
//
// Replaces (reference, /root/reference/acr/result_parser.py): CenterMap.parse_centermap_heatmap_
// adaptive_scale_batch :218-243 with K=1, nms :245-249, parameter_sampling :49-57, determine_coeff
// :42-47, parse_maps :85-190, parse :21-40 (+ rot6D_to_angular acr/utils.py:378-382).
//
// Three tiny kernels:
//   1. parse_top1   grid (B,2): 5x5 max-pool NMS + arg-max over the 64x64 centre map of one
//                   image/side (the reference runs maxpool + 2 topk + 3 gathers + where, with >=6
//                   device->host syncs).
//   2. parse_scan   1 CTA: stable compaction "left hands of all images, then right hands", the
//                   dummy-row rule for a side with no detection, the batch-global determine_coeff
//                   decision, counts.
//      parse_slot   (acr_b200_parse_per_frame instead of parse_scan) one thread per image: the
//                   fixed layout "row b = left hand of image b, row B+b = its right hand", each
//                   image parsed as the reference parses a batch of one.
//   3. parse_gather grid (2B): per output row gather 109 params at the centre (+106 prior values
//                   read at the OTHER hand's centre), split, 16 x rot6d->axis-angle.
#include "common.cuh"
#include "rotation.cuh"

namespace acr {

constexpr int MAPSZ = 64;
constexpr int NPIX = MAPSZ * MAPSZ;

struct ParseParams {
  acr_b200_map center[2], params[2], prior[2];
  int B;
  float thresh;
  const int64_t* meta_ids;
  const float* offsets;
  acr_b200_parse_out o;
  int32_t* row_src;  // (2B,4): image, side word, flat index, other side's flat index (or -1)
};

// side word of row_src: bit 0 = side; ROW_DUMMY marks a per-frame dummy row (its image has no detection on
// that side).  parse_scan never sets it: its dummy rows are recognised by the side's batch-wide count of 0.
constexpr int ROW_DUMMY = 2;

// determine_coeff (result_parser.py:42-47) on two flat centre indices: the cross-hand prior is kept iff the
// centres are at most 32 apart on the 64-grid ([y,x] distance in fp32, like the reference).
__device__ __forceinline__ bool centres_near(int il, int ir) {
  const float dy = (float)(il >> 6) - (float)(ir >> 6), dx = (float)(il & 63) - (float)(ir & 63);
  const float d = sqrtf(dy * dy + dx * dx);
  return !(d > 32.f);
}

__global__ void __launch_bounds__(256) parse_top1_kernel(ParseParams p) {
  __shared__ float s_map[NPIX];
  __shared__ float s_val[256];
  __shared__ int s_idx[256];
  const int b = blockIdx.x, side = blockIdx.y, t = threadIdx.x;
  const acr_b200_map cm = p.center[side];
  const float* src = cm.ptr + (size_t)b * NPIX * cm.pix_stride;
  for (int i = t; i < NPIX; i += 256) s_map[i] = src[(size_t)i * cm.pix_stride];
  __syncthreads();
  float best = -INFINITY;
  int besti = 0x7fffffff;
  for (int i = t; i < NPIX; i += 256) {
    const int y = i >> 6, x = i & 63;
    const float v = s_map[i];
    float mx = -INFINITY;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
      const int yy = y + dy;
      if (yy < 0 || yy >= MAPSZ) continue;
#pragma unroll
      for (int dx = -2; dx <= 2; ++dx) {
        const int xx = x + dx;
        if (xx < 0 || xx >= MAPSZ) continue;
        mx = fmaxf(mx, s_map[yy * MAPSZ + xx]);
      }
    }
    const float s = (mx == v) ? v : 0.f;  // det * (maxpool(det) == det)
    if (s > best || (s == best && i < besti)) { best = s; besti = i; }
  }
  s_val[t] = best; s_idx[t] = besti;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) {
      const float ov = s_val[t + w];
      const int oi = s_idx[t + w];
      if (ov > s_val[t] || (ov == s_val[t] && oi < s_idx[t])) { s_val[t] = ov; s_idx[t] = oi; }
    }
    __syncthreads();
  }
  if (t == 0) {
    p.o.top_idx[b * 2 + side] = s_idx[0];
    p.o.top_score[b * 2 + side] = s_val[0];
  }
}

// single CTA of 1024 threads; B is processed in strides
__global__ void __launch_bounds__(1024) parse_scan_kernel(ParseParams p) {
  __shared__ int s_cnt[2][1024];
  __shared__ int s_first[2];
  const int t = threadIdx.x, B = p.B;
  const int per = (B + 1023) / 1024;  // images per thread (contiguous => stable order)
  int c[2] = {0, 0};
  for (int i = 0; i < per; ++i) {
    const int b = t * per + i;
    if (b < B) {
      c[0] += p.o.top_score[b * 2 + 0] > p.thresh;
      c[1] += p.o.top_score[b * 2 + 1] > p.thresh;
    }
  }
  s_cnt[0][t] = c[0]; s_cnt[1][t] = c[1];
  if (t < 2) s_first[t] = 0x7fffffff;
  __syncthreads();
  // inclusive Hillis-Steele scan over 1024 partial counts, both sides at once
  for (int off = 1; off < 1024; off <<= 1) {
    int a0 = 0, a1 = 0;
    if (t >= off) { a0 = s_cnt[0][t - off]; a1 = s_cnt[1][t - off]; }
    __syncthreads();
    s_cnt[0][t] += a0; s_cnt[1][t] += a1;
    __syncthreads();
  }
  const int nl = s_cnt[0][1023], nr = s_cnt[1][1023];
  const int L = max(nl, 1), R = max(nr, 1);
  // first detection of each side (lowest image index)
  for (int i = 0; i < per; ++i) {
    const int b = t * per + i;
    if (b < B) {
      if (p.o.top_score[b * 2 + 0] > p.thresh) atomicMin(&s_first[0], b);
      if (p.o.top_score[b * 2 + 1] > p.thresh) atomicMin(&s_first[1], b);
    }
  }
  __syncthreads();
  // determine_coeff: distance between the first left and the first right centre of the batch
  bool prior_on = false;
  if (nl > 0 && nr > 0) prior_on = centres_near(p.o.top_idx[s_first[0] * 2 + 0], p.o.top_idx[s_first[1] * 2 + 1]);
  int pos[2] = {s_cnt[0][t] - c[0], s_cnt[1][t] - c[1]};  // exclusive prefix
  for (int i = 0; i < per; ++i) {
    const int b = t * per + i;
    if (b >= B) break;
    const bool dl = p.o.top_score[b * 2 + 0] > p.thresh, dr = p.o.top_score[b * 2 + 1] > p.thresh;
    if (dl) {
      int32_t* r = p.row_src + (size_t)(pos[0]++) * 4;
      r[0] = b; r[1] = 0; r[2] = p.o.top_idx[b * 2 + 0];
      r[3] = (dr && prior_on) ? p.o.top_idx[b * 2 + 1] : -1;
    }
    if (dr) {
      int32_t* r = p.row_src + (size_t)(L + pos[1]++) * 4;
      r[0] = b; r[1] = 1; r[2] = p.o.top_idx[b * 2 + 1];
      r[3] = (dl && prior_on) ? p.o.top_idx[b * 2 + 0] : -1;
    }
  }
  if (t == 0) {
    if (nl == 0) { int32_t* r = p.row_src; r[0] = 0; r[1] = 0; r[2] = 0; r[3] = -1; }
    if (nr == 0) { int32_t* r = p.row_src + (size_t)L * 4; r[0] = 0; r[1] = 1; r[2] = 0; r[3] = -1; }
    p.o.counts[0] = L; p.o.counts[1] = R; p.o.counts[2] = L + R; p.o.counts[3] = nl + nr;
    p.o.counts[4] = nl; p.o.counts[5] = nr;
  }
}

// Per-frame rows: image b alone is a batch of one for the reference, so a side it did not detect gets that
// batch's dummy row (pixel 0 of image b, no prior) and the prior is decided on image b's own pair.
// counts[3..5] are accumulated with atomics: the caller zeroes `counts` before the launch.
__global__ void __launch_bounds__(128) parse_slot_kernel(ParseParams p) {
  const int B = p.B, b = blockIdx.x * blockDim.x + threadIdx.x;
  bool dl = false, dr = false;
  if (b < B) {
    dl = p.o.top_score[b * 2 + 0] > p.thresh;
    dr = p.o.top_score[b * 2 + 1] > p.thresh;
    const int il = p.o.top_idx[b * 2 + 0], ir = p.o.top_idx[b * 2 + 1];
    const bool prior_on = dl && dr && centres_near(il, ir);
    int32_t* r = p.row_src + (size_t)b * 4;
    r[0] = b; r[1] = dl ? 0 : ROW_DUMMY; r[2] = dl ? il : 0; r[3] = prior_on ? ir : -1;
    r = p.row_src + (size_t)(B + b) * 4;
    r[0] = b; r[1] = dr ? 1 : 1 | ROW_DUMMY; r[2] = dr ? ir : 0; r[3] = prior_on ? il : -1;
  }
  const int nl = __popc(__ballot_sync(0xffffffffu, dl)), nr = __popc(__ballot_sync(0xffffffffu, dr));
  if ((threadIdx.x & 31) == 0 && (nl | nr)) {
    atomicAdd(&p.o.counts[3], nl + nr);
    atomicAdd(&p.o.counts[4], nl);
    atomicAdd(&p.o.counts[5], nr);
  }
  if (b == 0) { p.o.counts[0] = B; p.o.counts[1] = B; p.o.counts[2] = 2 * B; }
}

__global__ void __launch_bounds__(128) parse_gather_kernel(ParseParams p) {
  __shared__ float s_p[112];
  const int r = blockIdx.x, t = threadIdx.x;
  const int N = p.o.counts[2];
  if (r >= N) return;
  const int32_t* rs = p.row_src + (size_t)r * 4;
  const int b = rs[0], side = rs[1] & 1, fi = rs[2], ofi = rs[3];
  const bool real = !(rs[1] & ROW_DUMMY) && (side == 0 ? (p.o.counts[4] > 0) : (p.o.counts[5] > 0));
  if (t < 109) {
    const acr_b200_map pm = p.params[side];
    float v = pm.ptr[((size_t)b * NPIX + fi) * pm.pix_stride + t];
    if (ofi >= 0 && t >= 3) {
      const acr_b200_map pr = p.prior[side];  // own prior map, sampled at the other hand's centre
      v += pr.ptr[((size_t)b * NPIX + ofi) * pr.pix_stride + (t - 3)];
    }
    s_p[t] = v;
    p.o.params_pred[(size_t)r * 109 + t] = v;
    if (t < 3) p.o.cam[r * 3 + t] = v;
    if (t >= 99) p.o.betas[r * 10 + (t - 99)] = v;
  }
  __syncthreads();
  if (t < 16) {  // rotation t: 0 = global_orient (params 3..8), 1..15 = hand_pose (9..98)
    float aa[3];
    rot6d_to_aa(&s_p[3 + t * 6], aa);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      p.o.poses[(size_t)r * 48 + t * 3 + c] = aa[c];
      if (t == 0) p.o.global_orient[r * 3 + c] = aa[c];
      else p.o.hand_pose[(size_t)r * 45 + (t - 1) * 3 + c] = aa[c];
    }
  }
  if (t == 32) {
    p.o.detection_flag[r] = real ? 1.f : 0.f;
    p.o.batch_ids[r] = b;
    p.o.reorganize_idx[r] = p.meta_ids ? p.meta_ids[b] : (int64_t)b;
    p.o.centers_pred[r * 2 + 0] = fi & 63;
    p.o.centers_pred[r * 2 + 1] = fi >> 6;
    const acr_b200_map cm = p.center[side];
    p.o.centers_conf[r] = cm.ptr[((size_t)b * NPIX + fi) * cm.pix_stride];
    p.o.hand_type[r] = side;
  }
  if (p.offsets && p.o.offsets_out && t >= 64 && t < 74)
    p.o.offsets_out[(size_t)r * 10 + (t - 64)] = p.offsets[(size_t)b * 10 + (t - 64)];
}

}  // namespace acr

using namespace acr;

static int parse_launch(acr_b200_map l_center, acr_b200_map r_center, acr_b200_map l_params, acr_b200_map r_params,
                        acr_b200_map l_prior, acr_b200_map r_prior, int B, float conf_thresh,
                        const int64_t* meta_batch_ids, const float* offsets, acr_b200_parse_out out, bool per_frame,
                        cudaStream_t st) {
  ACR_CHECK_ARG(B > 0, "parse: B must be positive");
  ACR_CHECK_ARG(l_center.ptr && r_center.ptr && l_params.ptr && r_params.ptr && l_prior.ptr && r_prior.ptr,
                "parse: null map");
  ACR_CHECK_ARG(out.params_pred && out.cam && out.global_orient && out.hand_pose && out.betas && out.poses &&
                    out.detection_flag && out.reorganize_idx && out.batch_ids && out.centers_pred &&
                    out.centers_conf && out.hand_type && out.counts && out.top_idx && out.top_score && out.row_src,
                "parse: null output buffer");
  ParseParams p;
  p.center[0] = l_center; p.center[1] = r_center;
  p.params[0] = l_params; p.params[1] = r_params;
  p.prior[0] = l_prior; p.prior[1] = r_prior;
  p.B = B; p.thresh = conf_thresh; p.meta_ids = meta_batch_ids; p.offsets = offsets; p.o = out;
  p.row_src = out.row_src;
  parse_top1_kernel<<<dim3(B, 2), 256, 0, st>>>(p);
  ACR_CHECK_LAUNCH();
  if (per_frame) {
    ACR_CHECK_CUDA(cudaMemsetAsync(out.counts, 0, 8 * sizeof(int32_t), st));
    parse_slot_kernel<<<(B + 127) / 128, 128, 0, st>>>(p);
  } else {
    parse_scan_kernel<<<1, 1024, 0, st>>>(p);
  }
  ACR_CHECK_LAUNCH();
  parse_gather_kernel<<<2 * B, 128, 0, st>>>(p);
  ACR_CHECK_LAUNCH();
  return ACR_B200_OK;
}

extern "C" int acr_b200_parse(acr_b200_map l_center, acr_b200_map r_center, acr_b200_map l_params,
                              acr_b200_map r_params, acr_b200_map l_prior, acr_b200_map r_prior, int B,
                              float conf_thresh, const int64_t* meta_batch_ids, const float* offsets,
                              acr_b200_parse_out out, void* stream) {
  return parse_launch(l_center, r_center, l_params, r_params, l_prior, r_prior, B, conf_thresh, meta_batch_ids,
                      offsets, out, false, (cudaStream_t)stream);
}

extern "C" int acr_b200_parse_per_frame(acr_b200_map l_center, acr_b200_map r_center, acr_b200_map l_params,
                                        acr_b200_map r_params, acr_b200_map l_prior, acr_b200_map r_prior, int B,
                                        float conf_thresh, const int64_t* meta_batch_ids, const float* offsets,
                                        acr_b200_parse_out out, void* stream) {
  return parse_launch(l_center, r_center, l_params, r_params, l_prior, r_prior, B, conf_thresh, meta_batch_ids,
                      offsets, out, true, (cudaStream_t)stream);
}
