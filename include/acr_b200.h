/* acr_b200.h -- C ABI of the B200-native ACR hot path (libacr_b200.so).
 *
 * The reference (ZhengdiYu/Arbitrary-Hands-3D-Reconstruction) has no FFI of its own: its
 * boundary is a Python call surface (SURVEY.md section 8b).  Each entry point below names
 * the reference function(s) it replaces (path:line in /root/reference).  Conventions:
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked host;
 *   - `stream` is a cudaStream_t passed as void*; nothing synchronises, nothing allocates
 *     device memory (the caller owns all buffers and the plan arena);
 *   - return 0 on success, <0 on error; acr_b200_last_error() describes the last failure
 *     of the calling thread;
 *   - thread-compatible: concurrent calls must use different streams / plans.
 */
#ifndef ACR_B200_H_
#define ACR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACR_B200_OK 0
#define ACR_B200_EINVAL (-1)
#define ACR_B200_ECUDA (-2)
#define ACR_B200_ENOTSUP (-3)

const char* acr_b200_last_error(void);
/* "acr_b200 <version> sm_100a" */
const char* acr_b200_version(void);

/* ------------------------------------------------------------------------------------------
 * MANO
 * ---------------------------------------------------------------------------------------- */
/* Number of floats in one packed MANO model and the packing itself (host side, once per
 * asset).  Replaces the buffer registration of ManoLayer.__init__ (mano/manolayer.py:59-102)
 * plus MANOWrapper's left-hand shapedirs x-flip (acr/mano_wrapper.py:35, `flip_x`).
 * Inputs are HOST row-major fp32 arrays: shapedirs (778,3,10), posedirs (778,3,135),
 * v_template (778,3), j_regressor (16,778), weights (778,16), hands_mean (45).          */
size_t acr_b200_mano_model_floats(void);
int acr_b200_mano_pack_model(const float* shapedirs, const float* posedirs, const float* v_template,
                             const float* j_regressor, const float* weights, const float* hands_mean,
                             int flip_x, float* packed_host);

/* Fused MANO forward + weak-perspective projection for n hands.
 * Replaces ManoLayer.forward (mano/manolayer.py:104-276: Rodrigues :423-434, pose/shape blend
 * :175-182, joint regression :178, kinematic chain :187-223, LBS :226-240, tips/reorder/centre
 * :241-261), MANOWrapper.forward's two-layer dispatch (acr/mano_wrapper.py:40-46) and
 * batch_orth_proj / convert_kp2d_from_input_to_orgimg (acr/utils.py:384-397).
 *   model_l/model_r : packed models (device); either may be NULL if that side never occurs
 *   poses (n,48) axis-angle [root|hand] WITHOUT the mean pose; betas (n,10)
 *   hand_type (n) int32 0=left 1=right, or NULL => every row uses `default_side`
 *   n_dev : optional device int32; rows >= *n_dev are skipped (lets a CUDA graph run with
 *           the worst-case n = n_max and no host sync).  NULL => all n_max rows.
 *   center_idx : joint (after reordering) subtracted from joints and vertices, -1 = none
 *   cam (n,3) [s,tx,ty] and offsets (n,10) optional (NULL => projection outputs skipped)
 * Outputs (any may be NULL): verts (n,778,3), joints (n,21,3), center (n,3),
 *   verts_camed (n,778,3), pj2d (n,21,2), pj2d_org (n,21,2).                              */
int acr_b200_mano_forward(const float* model_l, const float* model_r, const float* poses,
                          const float* betas, const int32_t* hand_type, int default_side,
                          const int32_t* n_dev, int n_max, int center_idx, const float* cam,
                          const float* offsets, float* verts, float* joints, float* center,
                          float* verts_camed, float* pj2d, float* pj2d_org, void* stream);

/* Same kernel, with the vertex all-gather FUSED into it (replaces the gather step of nn.DataParallel,
 * acr/main.py:61 / the separate ncclAllGather of SURVEY.md 8e).  Besides the local outputs, every vertex is
 * stored straight into the gather buffers of ALL ranks over NVLink: 16-byte `multimem.st.v4.f32` through the
 * NVLS multicast mapping (the NVSwitch replicates the store) or, when `multicast_base` is 0, one 16-byte peer
 * store per rank.  The 8 int32 row counts of the shard (`counts_src`, as written by acr_b200_parse) travel the
 * same way, so the exchange needs no other collective.
 *
 * Symmetric allocation (identical layout on every rank, e.g. torch symmetric memory / CUDA IPC / VMM):
 *     [ slot 0 | slot 1 | flags ]          slot = verts[world][rows][778][3] fp32 at 0,
 *                                                 counts[world][8] int32 at counts_offset
 *     flags = uint64[world] at flags_offset (from the allocation base), zero-initialised.
 * Protocol (all device side, CUDA-graph safe; `local_state` = 16 zero-initialised device-local bytes holding
 * the step counter and a CTA counter):
 *   - launch number s (1,2,...) of this entry writes slot s & 1: rank r's rows land at rows [r*rows, (r+1)*rows)
 *     of that slot on every rank;
 *   - before touching the slot, the kernel waits until flags[q] >= s-1 for every rank q IN ITS OWN MEMORY: rank q
 *     publishes s-1 only at the end of its launch s-1, which it enqueued after consuming the data of step s-2
 *     (CONTRACT: a rank consumes step k's gathered data on the launching stream before its launch k+1) -- so the
 *     slot is free.  With two slots this dependency is a whole step old: ranks never wait for each other inside a
 *     step (no barrier), they can drift by up to one step;
 *   - the last CTA to finish publishes s into flags[rank] of every rank with a system-scope release store after
 *     a system-scope fence; acr_b200_gather_wait (stream-ordered, tiny) returns once flags[q] >= s for all q in
 *     this rank's memory, i.e. the data of step s from every rank has landed here.  Rows >= the shard's count
 *     keep older data: validity is counts[q][2].
 * `rows` (per rank and slot) must be even and >= n_max; every rank must launch every step.                      */
typedef struct acr_b200_gather {
  uint64_t peer_base[8];      /* base address of every rank's allocation, as mapped into THIS process     */
  uint64_t multicast_base;    /* NVLS multicast mapping of the allocation, or 0                            */
  int32_t world, rank;
  int64_t rows;
  uint64_t slot_bytes;        /* multiple of 16                                                            */
  uint64_t counts_offset;     /* inside a slot, multiple of 16, >= world*rows*778*3*4                      */
  uint64_t flags_offset;      /* from the allocation base, multiple of 16, >= 2*slot_bytes                 */
  void* local_state;          /* device-local, 16 bytes, zero-initialised once                             */
} acr_b200_gather;

int acr_b200_mano_forward_gather(const float* model_l, const float* model_r, const float* poses,
                                 const float* betas, const int32_t* hand_type, int default_side,
                                 const int32_t* n_dev, int n_max, int center_idx, const float* cam,
                                 const float* offsets, float* verts, float* joints, float* center,
                                 float* verts_camed, float* pj2d, float* pj2d_org,
                                 const int32_t* counts_src, const acr_b200_gather* gather, void* stream);
/* Stream-ordered wait until the most recent gather launch of EVERY rank has landed in this rank's buffer. */
int acr_b200_gather_wait(const acr_b200_gather* gather, void* stream);

/* Camera translation of every hand from its 21 joints: the closed-form weighted least squares of
 * estimate_translation_np (acr/utils.py:430-472) -- the reference's own fall-back for the host-side
 * cv2.solvePnPRansac loop (estimate_translation :474-519, called from vertices_kp3d_projection :403-407,
 * SURVEY.md 8f-1).  joints_2d = (pj2d+1)*img_size/2 as in :404; a joint is used iff its pixel y > -2
 * and its z != -2 (:489-492); fewer than 4 usable joints -> (-1,-1,-1).  fp64 normal equations.
 * j3d (n,21,3), pj2d (n,21,2) -> cam_trans (n,3).  n_dev as in acr_b200_mano_forward.              */
int acr_b200_cam_trans(const float* j3d, const float* pj2d, const int32_t* n_dev, int n_max, float focal_length,
                       float img_size, float* cam_trans, void* stream);

/* Frame pre-processing on the device (SURVEY.md 8f-2): n BGR frames (n,H,W,3) -> RGB, white (255) pad to a
 * `side` x `side` square (pad_t rows above, pad_l columns left), bicubic resize to out_size x out_size.
 * Replaces img_preprocess / process_image_ori / image_pad_white_bg + cv2.resize(INTER_CUBIC)
 * (acr/utils.py:1303-1337).  Integer arithmetic of OpenCV's generic 8-bit cubic path (11-bit coefficients,
 * replicate border, (sum + 2^21) >> 22); the (out_size,4) int16 coefficient and (out_size) int32 offset
 * tables come from acr_b200/preprocess.py::cubic_tables (host, float32 like OpenCV).                   */
int acr_b200_preprocess(const uint8_t* frames_bgr, int n, int H, int W, const int16_t* coef_x,
                        const int32_t* ofs_x, const int16_t* coef_y, const int32_t* ofs_y, int side, int pad_t,
                        int pad_l, int out_size, uint8_t* out_rgb, void* stream);

/* Temporal OneEuro smoothing of poses / betas between parse and MANO, in place, on the device
 * (SURVEY.md 8f-3).  Replaces OneEuroFilter / LowPassFilter (acr/utils.py:1485-1527), smooth_results
 * (:1478-1482), smooth_global_rot_matrix (:1466-1470) and the per-frame host loop of acr/main.py:69-83.
 * `state`: device buffer of acr_b200_one_euro_state_floats() floats, zero-initialised = "no history";
 * one filter bank per hand type (0 left, 1 right), like the reference's filter_dict -- i.e. for streaming
 * one frame at a time (the reference asserts exactly two rows).  Rows with detection_flag == 0 are skipped.
 * poses (n,48) and betas (n,10) are updated in place.                                              */
size_t acr_b200_one_euro_state_floats(void);
int acr_b200_one_euro_smooth(float* poses, float* betas, const int32_t* hand_type, const float* detection_flag,
                             const int32_t* n_dev, int n_max, float* state, float smooth_coeff, void* stream);

/* The same filter for many independent video streams in one launch (one row per hand, any number of slots).
 * `state`: n_streams consecutive blocks of acr_b200_one_euro_state_floats() floats; block s is stream s's
 * history, laid out exactly like the single-stream state above (zeroing block s on the launching stream
 * resets stream s: "new clip").  The bank of row r is (stream_ids[batch_ids[r]], hand_type[r]):
 *   batch_ids (n) int64   slot of each row (acr_b200_parse / _per_frame write it)
 *   stream_ids (B) int32  stream of each slot; a slot whose id is outside [0, n_streams), e.g. -1 for a
 *                         padding slot, is not filtered and leaves every state block untouched.
 * Rows with detection_flag == 0 are skipped as above.  CONTRACT: the non-negative stream ids of one call are
 * distinct -- two slots of the same stream in one launch would race on its state.  hand_type, batch_ids and
 * stream_ids are required.  acr_b200_one_euro_smooth is this kernel with one stream and the bank = hand type. */
int acr_b200_one_euro_smooth_streams(float* poses, float* betas, const int32_t* hand_type,
                                     const float* detection_flag, const int64_t* batch_ids,
                                     const int32_t* stream_ids, int n_streams, const int32_t* n_dev, int n_max,
                                     float* state, float smooth_coeff, void* stream);

/* ------------------------------------------------------------------------------------------
 * Rotations
 * ---------------------------------------------------------------------------------------- */
/* rot6D_to_angular (acr/utils.py:378-382): n_rot 6-vectors -> n_rot axis-angle 3-vectors,
 * through Gram-Schmidt (:362-376), 4-case quaternion (:826-906), atan2 (:773-823), NaN->0. */
int acr_b200_rot6d_to_aa(const float* rot6d, int n_rot, float* aa, void* stream);
/* batch_rodrigues (mano/manolayer.py:423-434): n axis-angle -> n row-major 3x3.            */
int acr_b200_rodrigues(const float* aa, int n_rot, float* rotmat, void* stream);

/* ------------------------------------------------------------------------------------------
 * Centre parsing + parameter sampling
 * ---------------------------------------------------------------------------------------- */
typedef struct acr_b200_map {      /* one fp32 NHWC map: element (b,y,x,c) at              */
  const float* ptr;                /* ptr[((b*H + y)*W + x)*pix_stride + c]                */
  int pix_stride;
} acr_b200_map;

typedef struct acr_b200_parse_out {
  /* compacted rows, left hands first (all images in order) then right hands; capacity 2*B
   * (acr_b200_parse_per_frame: fixed rows, see there)                                     */
  float* params_pred;        /* (2B,109) */
  float* cam;                /* (2B,3)   */
  float* global_orient;      /* (2B,3)   axis-angle */
  float* hand_pose;          /* (2B,45)  axis-angle */
  float* betas;              /* (2B,10)  */
  float* poses;              /* (2B,48)  = [global_orient | hand_pose] */
  float* detection_flag;     /* (2B)     1.0 / 0.0 */
  int64_t* reorganize_idx;   /* (2B)     meta batch id of the row's image */
  int64_t* batch_ids;        /* (2B)     local image index of the row */
  int64_t* centers_pred;     /* (2B,2)   [x,y] on the 64-grid, rows as above */
  float* centers_conf;       /* (2B)     raw centre-map value at the centre */
  int32_t* hand_type;        /* (2B)     0 left, 1 right */
  float* offsets_out;        /* (2B,10)  offsets row of the image, or NULL */
  int32_t* counts;           /* (8) [0]=L, [1]=R, [2]=L+R, [3]=#true detections, [4]=#left, [5]=#right */
  /* dense per-image scratch, (B,2): flat index and score of the top-1 centre of each side */
  int32_t* top_idx;
  float* top_score;
  int32_t* row_src;          /* (2B,4) scratch: image, side (| 2: per-frame dummy row), flat index, other side's index | -1 */
} acr_b200_parse_out;

/* ResultParser.parse (acr/result_parser.py:21-40) = parse_maps (:85-190) with K=1 centre
 * extraction (:218-249), parameter sampling (:49-57), cross-hand prior (:141-145) gated by
 * determine_coeff (:42-47), then rot6D_to_angular on global_orient / hand_pose.
 * B images, H=W=64 maps.  meta_batch_ids (B) int64 may be NULL (=> arange), offsets (B,10)
 * may be NULL.  All batch>1 quirks of the reference are reproduced (see oracle/parse_ref.py). */
int acr_b200_parse(acr_b200_map l_center, acr_b200_map r_center, acr_b200_map l_params,
                   acr_b200_map r_params, acr_b200_map l_prior, acr_b200_map r_prior, int B,
                   float conf_thresh, const int64_t* meta_batch_ids, const float* offsets,
                   acr_b200_parse_out out, void* stream);

/* Per-frame parse: every image b is parsed exactly as the reference's ResultParser.parse parses that image
 * alone (a batch of one), so a row never depends on the other images of the batch -- the semantics of B
 * independent video streams.  Same arguments and output struct as acr_b200_parse, but a FIXED layout, no
 * compaction: row b is image b's left hand, row B+b its right hand, counts = [B, B, 2B, #true, #left, #right].
 *   - a side not detected in image b gets the reference's batch-of-one dummy row: sampled at pixel 0 of
 *     image b, no prior, detection_flag 0, hand_type = that side, reorganize_idx = meta_batch_ids[b];
 *   - the cross-hand prior is applied iff image b detected both hands and their centres are at most 32 apart
 *     on the 64-grid (determine_coeff evaluated on image b).
 * One thread per image replaces acr_b200_parse's one-CTA batch scan.                                  */
int acr_b200_parse_per_frame(acr_b200_map l_center, acr_b200_map r_center, acr_b200_map l_params,
                             acr_b200_map r_params, acr_b200_map l_prior, acr_b200_map r_prior, int B,
                             float conf_thresh, const int64_t* meta_batch_ids, const float* offsets,
                             acr_b200_parse_out out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Network launch plan (backbone + heads)
 * ---------------------------------------------------------------------------------------- */
enum {
  ACR_OP_STEM = 1,        /* uint8 NHWC image -> x/255*2-1 -> conv3x3 s2 + BN + ReLU           */
  ACR_OP_CONV = 2,        /* implicit-GEMM NHWC conv (k in {1,3}, s in {1,2}) on tcgen05        */
  ACR_OP_FUSE = 3,        /* relu(sum_i nearest_up(term_i, 2^shift_i)), fp32 accumulation       */
  ACR_OP_BILINEAR2X = 4,  /* F.interpolate(x2, bilinear, align_corners=True)                    */
  ACR_OP_COORD = 5,       /* write the two coord-conv channels                                  */
  ACR_OP_POOL = 6,        /* Hadamard_product: softmax over HW x feature matmul (partials)      */
  ACR_OP_PARTHEAD = 7,    /* merge partials + LocallyConnected2d + Linear + per-image bias      */
  ACR_OP_CONV_REF = 8,    /* debug: same contract as ACR_OP_CONV on CUDA cores (tests only)     */
  ACR_OP_FINALCONV = 9,   /* (retired)                                                          */
  ACR_OP_IM2COL_STEM = 10, /* uint8 NHWC image -> 3x3 s2 im2col of x/255*2-1, 27(+5 zero) 16-bit channels */
  ACR_OP_STEM_TC = 11      /* STEM on the tensor cores: the im2col operand is built in shared memory, never in HBM   */
};
enum { ACR_CONV_BIAS_PER_IMAGE = 1, ACR_CONV_POW11_CH0 = 2, ACR_CONV_XPAIR = 4, ACR_CONV_S2X = 8, ACR_CONV_EXTRA = 16 };
enum { ACR_DT_BF16 = 0, ACR_DT_F16 = 1, ACR_DT_F32 = 2, ACR_DT_U8 = 3 };

typedef struct acr_b200_tensor {  /* NHWC activation inside the arena (per-image extents)  */
  uint64_t offset;                /* byte offset of element (0,0,0,0) from the arena base   */
  int32_t C, H, W;                /* logical channels (multiple of 8 for 16-bit types)      */
  int32_t pix_stride;             /* elements between neighbouring pixels (>= C)            */
  int32_t dtype;
  int32_t external;               /* 1: `offset` is relative to the external-input pointer  */
} acr_b200_tensor;

/* One launch.  Which fields are read depends on `kind`:
 *  STEM      in[0]=image(u8,external) out; w_offset[0]=fp32 [27][64] folded weights, [1]=fp32 bias[64]
 *  STEM_TC   in[0]=image(u8,external) out (64 ch, H/2 x W/2, 16-bit); w_offset[0]=packed [64][32] 16-bit weights (input
 *            channel (ky*3+kx)*3+ci, 27..31 zero, BN folded), [1]=fp32 bias[64]: conv1 + bn1 + ReLU of acr/model.py:832-835
 *            as one tcgen05 GEMM whose A operand (the 27 normalised taps of every output pixel) is built in shared memory
 *  IM2COL_STEM in[0]=image(u8,external) out (32 ch, H/2 x W/2): channel (ky*3+kx)*3+ci = normalised tap,
 *            0 outside the image; the stem conv then runs as a 1x1 CONV on the tensor cores
 *  CONV(_REF) in[0]=x, in[1]=residual (has_residual) out; w_offset[0]=packed 16-bit weights
 *            [cout_pad][k*k][cin_pad], w_offset[1]=fp32 bias[cout_pad]; shift[0] = flag bits:
 *            ACR_CONV_BIAS_PER_IMAGE (bias = fp32 (B,cout_pad) tensor aux[0] in the arena instead of
 *            w_offset[1]) | ACR_CONV_POW11_CH0 (output channel 0 -> 1.1**x, acr/model.py:95-96)
 *            | ACR_CONV_XPAIR (3x3 s1 64->64 whose weights are the x-paired expansion of a 32->32 conv: channel =
 *            (x parity)*32 + c on a W/2 grid; the kx=0 / kx=2 taps are non-zero only in the [N 0..31][K 32..63] /
 *            [N 32..63][K 0..31] corner, which is all the kernel multiplies)
 *            | ACR_CONV_EXTRA (in[1..n_in) are further terms of the same shape class as `out`, term j nearest-upsampled by
 *            2**shift[j]: out = act(conv(in[0]) + bias + sum of terms) -- the fuse sum of HighResolutionModule.forward
 *            (acr/model.py:677-684) folded into the conv that produces one of its terms; no residual then)
 *            | ACR_CONV_S2X (3x3 STRIDE-2 conv of a dense 32-channel tensor: in[0] is its x-paired view (H, W/2, 64) --
 *            even pixel's channels then the odd neighbour's in one 128-byte row -- `out` is (H/2, W/2); the packed
 *            weights [cout_pad][9][64] carry the 32 input channels of tap (ky,kx) at K offset 32*(kx != 1))
 *  FUSE      in[0..n_in) with shift[i]; out
 *  BILINEAR2X / COORD (fparam unused; COORD writes channels [in[0].C, pix_stride) of `out`)
 *  POOL      in[0]=contact features (256ch), in[1]=segm logits; out = partials (fp32, 1x1xC)
 *  PARTHEAD  in[0]=partials; out=pooled (fp32 256*32); aux[0..1]=bias_img l,r (112); aux[2..3]=
 *            pare l,r (106); w_offset[0..1]=LC weights l,r; [2],[3]=shape conv w,b; [4..5]=Linear w
 *            l,r; [6..7]=Linear b; [8..9]=final conv w (109,218) l,r; [10..11]=final conv b
 *  FINALCONV (retired: the folded contact_layers[4|5] conv now runs as a CONV with
 *            ACR_CONV_BIAS_PER_IMAGE on the tensor cores)                                  */
typedef struct acr_b200_op {
  int32_t kind;
  int32_t n_in;
  acr_b200_tensor out;
  acr_b200_tensor in[4];
  acr_b200_tensor aux[4];
  uint64_t w_offset[12];          /* byte offsets into the weight blob                      */
  int32_t k, stride, relu, has_residual;
  int32_t cin_pad, cout_pad;      /* K per tap / N, multiples of 16                         */
  int32_t shift[4];
  int32_t stream_id;              /* plan-internal stream (branch-level concurrency)        */
  int32_t wait_mask;              /* bit i: wait for the last op recorded on stream i       */
  float fparam[4];
} acr_b200_op;

typedef struct acr_b200_plan acr_b200_plan;

/* Build a launch plan for `batch` images.  `arena` (device, `arena_bytes`) holds every
 * activation; `weights` (device) the packed weight blob; ops are copied.  Creates the TMA
 * tensor maps and internal streams/events.  Replaces the module tree construction +
 * forward dispatch of acr/model.py:23-65 (ACR), :691-865 (HigherResolutionNet).           */
int acr_b200_plan_create(const acr_b200_op* ops, int n_ops, int batch, void* arena,
                         size_t arena_bytes, const void* weights, size_t weight_bytes,
                         int act_dtype, acr_b200_plan** plan_out);
/* Run the plan on `stream`: `image` is the external uint8 (batch,512,512,3) input.        */
int acr_b200_plan_run(acr_b200_plan* plan, const void* image, void* stream);
/* Like plan_run, but brackets every launch with CUDA events on `stream` (serialising the plan) and
 * accumulates device milliseconds / launch counts per op kind into ms_by_kind[16] / n_by_kind[16]
 * (host arrays, indexed by ACR_OP_*).  Synchronises `stream`.  Used by bench.py for the roofline. */
int acr_b200_plan_profile(acr_b200_plan* plan, const void* image, void* stream, float* ms_by_kind,
                          int32_t* n_by_kind);
/* Number of kernel launches one plan_run issues (for bench.py's gpu_launches).            */
int acr_b200_plan_num_launches(const acr_b200_plan* plan);
void acr_b200_plan_destroy(acr_b200_plan* plan);

/* Single-op entry used by the parity tests (same code path as inside a plan).             */
int acr_b200_run_op(const acr_b200_op* op, int batch, void* arena, const void* weights,
                    const void* external, int act_dtype, void* stream);

/* Which kernel instance and schedule an ACR_OP_CONV launch gets (tests: proves what a case exercised).
 * Builds the conv's plan exactly as plan_create / run_op do (same environment switches), writes the first
 * n_info of the fields below to `info` (host) and frees the plan; nothing is launched.  Encoding the TMA
 * tensor maps needs the CUDA driver, so this fails on a machine without one.
 *   CK          channel chunk of the K loop (16 / 32 / 64)
 *   MODE        template bits of the instance: 1 PATCH, 2 RESIDENT, 4 XPAIR, 8 DIAG, 16 P1, 32 S2X
 *   B_RESIDENT  weights resident in shared memory for the whole kernel
 *   NSPLIT/NSUB each 16x16 super-tile is NSPLIT virtual tiles of NSUB output channels
 *   NBUF        TMEM accumulator buffers (2 = the epilogue of one tile overlaps the MMAs of the next)
 *   EPILOGUE    0 direct stores, 1 staged (per-warp slabs, TMA residual loads + TMA stores), 2 TMA store
 *   EPI_NB      slab buffers per epilogue warp of the staged epilogue
 *   SA/SB       A / B operand stages (SB = 0: resident weights)
 *   GRID        persistent CTAs = min(VTILES, SMs, ACR_B200_CONV_MAX_CTAS if set)
 *   VTILES      virtual tiles of the launch (super-tiles of all images x NSPLIT)                  */
enum {
  ACR_CONV_INFO_CK, ACR_CONV_INFO_MODE, ACR_CONV_INFO_B_RESIDENT, ACR_CONV_INFO_NSPLIT, ACR_CONV_INFO_NSUB,
  ACR_CONV_INFO_NBUF, ACR_CONV_INFO_EPILOGUE, ACR_CONV_INFO_EPI_NB, ACR_CONV_INFO_SA, ACR_CONV_INFO_SB,
  ACR_CONV_INFO_GRID, ACR_CONV_INFO_VTILES, ACR_CONV_INFO_N
};
int acr_b200_conv_describe(const acr_b200_op* op, int batch, void* arena, const void* weights,
                           int act_dtype, int32_t* info, int n_info);

/* Host-side weight folding/packing for one conv (acr_b200_weights_pack of SURVEY.md 8b):
 * folds eval-mode BatchNorm (acr/model.py BN after every conv) into w/b and repacks
 * OIHW fp32 -> [cout_pad][kh][kw][cin_pad] 16-bit (K-major rows for the UMMA B operand).
 * bn_* may be NULL (no BN); conv_bias may be NULL.  All pointers are HOST pointers.       */
int acr_b200_pack_conv(const float* w_oihw, const float* conv_bias, const float* bn_gamma,
                       const float* bn_beta, const float* bn_mean, const float* bn_var, float bn_eps,
                       int cout, int cin, int k, int cout_pad, int cin_pad, int act_dtype,
                       void* w_packed_host, float* bias_host);

#ifdef __cplusplus
}
#endif
#endif /* ACR_B200_H_ */
