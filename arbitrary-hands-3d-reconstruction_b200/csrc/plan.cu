// Launch plan: the network as a flat list of kernel launches over one activation arena.
// Replaces the nn.Module tree walk of the reference (acr/model.py:32-65 ACR.forward/head_forward,
// :831-865 HigherResolutionNet.forward, :668-686 HighResolutionModule.forward) with a precompiled
// schedule: tensor maps built once, branch-level concurrency on plan-internal streams, no Python
// in the loop.  Also hosts the BN-folding weight packer.
#include <stdlib.h>
#include <new>
#include <vector>

#include "ops.cuh"

namespace acr {

static TensorRef resolve(const acr_b200_tensor& t, char* arena, const char* external) {
  TensorRef r;
  r.ptr = (t.external ? const_cast<char*>(external) : arena) + t.offset;
  r.C = t.C; r.H = t.H; r.W = t.W; r.pix_stride = t.pix_stride; r.dtype = t.dtype;
  return r;
}

static int make_conv_args(const acr_b200_op& op, int batch, char* arena, const char* weights,
                          const char* external, ConvArgs* a) {
  ACR_CHECK_ARG(op.n_in >= 1, "conv: missing input");
  a->in = resolve(op.in[0], arena, external);
  a->out = resolve(op.out, arena, external);
  a->has_res = op.has_residual;
  if (op.has_residual) {
    ACR_CHECK_ARG(op.n_in >= 2, "conv: residual flagged but in[1] missing");
    a->res = resolve(op.in[1], arena, external);
    ACR_CHECK_ARG(a->res.H == a->out.H && a->res.W == a->out.W, "conv: residual shape mismatch");
  } else {
    a->res = a->out;
  }
  a->w = weights + op.w_offset[0];
  a->bias = reinterpret_cast<const float*>(weights + op.w_offset[1]);
  a->k = op.k; a->stride = op.stride; a->relu = op.relu;
  a->cin_pad = op.cin_pad; a->cout_pad = op.cout_pad; a->batch = batch;
  a->bias_per_image = (op.shift[0] & ACR_CONV_BIAS_PER_IMAGE) ? 1 : 0;
  a->pow11_ch0 = (op.shift[0] & ACR_CONV_POW11_CH0) ? 1 : 0;
  a->xpair = (op.shift[0] & ACR_CONV_XPAIR) ? 1 : 0;
  a->s2x = (op.shift[0] & ACR_CONV_S2X) ? 1 : 0;
  a->n_ext = 0;
  if (op.shift[0] & ACR_CONV_EXTRA) {
    ACR_CHECK_ARG(!op.has_residual && op.n_in >= 2 && op.n_in <= 4, "conv: extra terms need 2..4 inputs and no residual");
    a->n_ext = op.n_in - 1;
    for (int e = 0; e < a->n_ext; ++e) {
      a->ext[e] = resolve(op.in[e + 1], arena, external);
      a->ext_shift[e] = op.shift[e + 1];
      ACR_CHECK_ARG(a->ext_shift[e] >= 0 && a->ext_shift[e] <= 3 && (a->ext[e].H << a->ext_shift[e]) == a->out.H &&
                        (a->ext[e].W << a->ext_shift[e]) == a->out.W && a->ext[e].C == a->out.C && a->ext[e].dtype == a->out.dtype,
                    "conv: extra term %d shape mismatch", e);
    }
  }
  if (a->bias_per_image) {
    ACR_CHECK_ARG(op.aux[0].dtype == ACR_DT_F32 && op.aux[0].pix_stride >= op.cout_pad, "conv: per-image bias tensor (aux[0]) malformed");
    a->bias = reinterpret_cast<const float*>(arena + op.aux[0].offset);
  }
  ACR_CHECK_ARG((op.k == 1 || op.k == 3) && (op.stride == 1 || op.stride == 2), "conv: k/stride unsupported");
  if (a->s2x) ACR_CHECK_ARG(op.stride == 2 && a->out.H * 2 == a->in.H && a->out.W == a->in.W, "conv: x-paired stride-2 spatial mismatch");
  else ACR_CHECK_ARG(a->out.H * op.stride == a->in.H && a->out.W * op.stride == a->in.W, "conv: spatial mismatch");
  ACR_CHECK_ARG(op.cout_pad % 16 == 0 && op.cin_pad % 16 == 0 && op.cout_pad <= 1024, "conv: padded channel counts");
  ACR_CHECK_ARG(a->out.pix_stride >= op.cout_pad, "conv: output buffer narrower than cout_pad");
  return ACR_B200_OK;
}

// fp32 validation plan: every op on the fp32-storage / fp64-accumulate kernels of validate_f32.cu
static int run_one_f32(const acr_b200_op& op, int batch, char* arena, const char* weights, const char* external,
                       cudaStream_t st) {
  switch (op.kind) {
    case ACR_OP_STEM:
      ACR_CHECK_ARG(external != nullptr, "stem: external image pointer is null");
      return launch_stem_f32(resolve(op.in[0], arena, external), resolve(op.out, arena, external),
                             reinterpret_cast<const float*>(weights + op.w_offset[0]),
                             reinterpret_cast<const float*>(weights + op.w_offset[1]), batch, st);
    case ACR_OP_CONV:
    case ACR_OP_CONV_REF: {
      ConvArgs a;
      int rc = make_conv_args(op, batch, arena, weights, external, &a);
      if (rc) return rc;
      return launch_conv_f32(a, st);
    }
    case ACR_OP_FUSE: {
      FuseArgs f;
      f.out = resolve(op.out, arena, external);
      f.n_in = op.n_in; f.relu = op.relu; f.batch = batch;
      ACR_CHECK_ARG(op.n_in >= 1 && op.n_in <= 4, "fuse: n_in");
      for (int i = 0; i < op.n_in; ++i) { f.in[i] = resolve(op.in[i], arena, external); f.shift[i] = op.shift[i]; }
      return launch_fuse_f32(f, st);
    }
    case ACR_OP_BILINEAR2X:
      return launch_bilinear2x_f32(resolve(op.in[0], arena, external), resolve(op.out, arena, external), batch, st);
    case ACR_OP_COORD:
      return launch_coord_f32(resolve(op.out, arena, external), op.in[0].C, batch, st);
    case ACR_OP_POOL:
      return launch_pool_f32(resolve(op.in[0], arena, external), resolve(op.in[1], arena, external),
                             reinterpret_cast<float*>(arena + op.out.offset), batch, st);
    default:
      set_error("op kind %d has no fp32 validation kernel", op.kind);
      return ACR_B200_EINVAL;
  }
}

static int run_one(const acr_b200_op& op, int batch, char* arena, const char* weights, const char* external,
                   int act_dtype, const ConvTcPlan* tc, cudaStream_t st) {
  if (act_dtype == ACR_DT_F32 && op.kind != ACR_OP_PARTHEAD) return run_one_f32(op, batch, arena, weights, external, st);
  switch (op.kind) {
    case ACR_OP_STEM: {
      ACR_CHECK_ARG(external != nullptr, "stem: external image pointer is null");
      return launch_stem(resolve(op.in[0], arena, external), resolve(op.out, arena, external),
                         reinterpret_cast<const float*>(weights + op.w_offset[0]),
                         reinterpret_cast<const float*>(weights + op.w_offset[1]), batch, act_dtype, st);
    }
    case ACR_OP_STEM_TC:
      ACR_CHECK_ARG(external != nullptr, "stem_tc: external image pointer is null");
      return launch_stem_tc(resolve(op.in[0], arena, external), resolve(op.out, arena, external), weights + op.w_offset[0],
                            reinterpret_cast<const float*>(weights + op.w_offset[1]), batch, act_dtype, st);
    case ACR_OP_IM2COL_STEM:
      ACR_CHECK_ARG(external != nullptr, "im2col_stem: external image pointer is null");
      return launch_im2col_stem(resolve(op.in[0], arena, external), resolve(op.out, arena, external), batch, act_dtype, st);
    case ACR_OP_CONV: {
      if (tc) return conv_tc_launch(tc, st);
      ConvArgs a;
      int rc = make_conv_args(op, batch, arena, weights, external, &a);
      if (rc) return rc;
      ConvTcPlan* tmp = nullptr;
      rc = conv_tc_prepare(a, act_dtype, &tmp);
      if (rc) return rc;
      rc = conv_tc_launch(tmp, st);
      conv_tc_free(tmp);
      return rc;
    }
    case ACR_OP_CONV_REF: {
      ConvArgs a;
      int rc = make_conv_args(op, batch, arena, weights, external, &a);
      if (rc) return rc;
      return launch_conv_ref(a, act_dtype, st);
    }
    case ACR_OP_FUSE: {
      FuseArgs f;
      f.out = resolve(op.out, arena, external);
      f.n_in = op.n_in; f.relu = op.relu; f.batch = batch;
      ACR_CHECK_ARG(op.n_in >= 1 && op.n_in <= 4, "fuse: n_in");
      for (int i = 0; i < op.n_in; ++i) { f.in[i] = resolve(op.in[i], arena, external); f.shift[i] = op.shift[i]; }
      return launch_fuse(f, act_dtype, st);
    }
    case ACR_OP_BILINEAR2X:
      return launch_bilinear2x(resolve(op.in[0], arena, external), resolve(op.out, arena, external), batch, act_dtype, st);
    case ACR_OP_COORD:
      return launch_coord(resolve(op.out, arena, external), op.in[0].C, batch, act_dtype, st);
    case ACR_OP_POOL:
      return launch_pool(resolve(op.in[0], arena, external), resolve(op.in[1], arena, external),
                         reinterpret_cast<float*>(arena + op.out.offset), batch, act_dtype, st);
    case ACR_OP_PARTHEAD: {
      PartHeadArgs a;
      a.part = reinterpret_cast<const float*>(arena + op.in[0].offset);
      a.pooled = reinterpret_cast<float*>(arena + op.out.offset);
      auto W = [&](int i) { return reinterpret_cast<const float*>(weights + op.w_offset[i]); };
      a.lc_w[0] = W(0); a.lc_w[1] = W(1); a.shape_w = W(2); a.shape_b = W(3);
      a.lin_w[0] = W(4); a.lin_w[1] = W(5); a.lin_b[0] = W(6); a.lin_b[1] = W(7);
      a.fin_w[0] = W(8); a.fin_w[1] = W(9); a.fin_b[0] = W(10); a.fin_b[1] = W(11);
      a.bias_img[0] = reinterpret_cast<float*>(arena + op.aux[0].offset);
      a.bias_img[1] = reinterpret_cast<float*>(arena + op.aux[1].offset);
      a.pare[0] = reinterpret_cast<float*>(arena + op.aux[2].offset);
      a.pare[1] = reinterpret_cast<float*>(arena + op.aux[3].offset);
      a.batch = batch;
      return launch_parthead(a, st);
    }
    default:
      set_error("unknown op kind %d", op.kind);
      return ACR_B200_EINVAL;
  }
}

}  // namespace acr

using namespace acr;

constexpr int MAX_STREAMS = 8;

struct acr_b200_plan {
  std::vector<acr_b200_op> ops;
  std::vector<ConvTcPlan*> tc;
  int batch = 0, act_dtype = 0, n_streams = 1;
  char* arena = nullptr;
  size_t arena_bytes = 0;
  const char* weights = nullptr;
  cudaStream_t streams[MAX_STREAMS] = {};
  std::vector<cudaEvent_t> ev_op;      // one event per op (recorded when some later op waits on its stream)
  cudaEvent_t ev_begin = nullptr;
};

extern "C" int acr_b200_plan_create(const acr_b200_op* ops, int n_ops, int batch, void* arena,
                                    size_t arena_bytes, const void* weights, size_t weight_bytes,
                                    int act_dtype, acr_b200_plan** plan_out) {
  ACR_CHECK_ARG(ops && n_ops > 0 && batch > 0 && arena && weights && plan_out, "plan_create: bad arguments");
  ACR_CHECK_ARG(act_dtype == ACR_DT_BF16 || act_dtype == ACR_DT_F16 || act_dtype == ACR_DT_F32,
                "plan_create: act_dtype must be bf16/f16 (product) or f32 (validation plan)");
  acr_b200_plan* p = new (std::nothrow) acr_b200_plan();
  ACR_CHECK_ARG(p != nullptr, "plan_create: out of host memory");
  p->ops.assign(ops, ops + n_ops);
  p->tc.assign(n_ops, nullptr);
  p->batch = batch; p->act_dtype = act_dtype;
  p->arena = static_cast<char*>(arena); p->arena_bytes = arena_bytes;
  p->weights = static_cast<const char*>(weights);
  (void)weight_bytes;
  int rc = ACR_B200_OK;
  for (int i = 0; i < n_ops && rc == ACR_B200_OK; ++i) {
    const acr_b200_op& op = p->ops[i];
    if (op.stream_id < 0 || op.stream_id >= MAX_STREAMS) { set_error("op %d: stream_id out of range", i); rc = ACR_B200_EINVAL; break; }
    if (op.stream_id + 1 > p->n_streams) p->n_streams = op.stream_id + 1;
    if (!op.out.external && op.kind != ACR_OP_COORD) {
      const size_t esz = op.out.dtype == ACR_DT_F32 ? 4 : (op.out.dtype == ACR_DT_U8 ? 1 : 2);
      const size_t need = op.out.offset + (size_t)batch * op.out.H * op.out.W * op.out.pix_stride * esz;
      if (need > arena_bytes) { set_error("op %d: output exceeds the arena (%zu > %zu)", i, need, arena_bytes); rc = ACR_B200_EINVAL; break; }
    }
    if (op.kind == ACR_OP_CONV && act_dtype != ACR_DT_F32) {
      ConvArgs a;
      rc = make_conv_args(op, batch, p->arena, p->weights, nullptr, &a);
      if (rc == ACR_B200_OK) rc = conv_tc_prepare(a, act_dtype, &p->tc[i]);
    }
  }
  if (rc == ACR_B200_OK) {
    for (int s = 1; s < p->n_streams && rc == ACR_B200_OK; ++s)
      if (cudaStreamCreateWithFlags(&p->streams[s], cudaStreamNonBlocking) != cudaSuccess) { set_error("plan_create: cudaStreamCreate failed"); rc = ACR_B200_ECUDA; }
    p->ev_op.assign(n_ops, nullptr);
    if (p->n_streams > 1) {
      for (int i = 0; i < n_ops && rc == ACR_B200_OK; ++i)
        if (cudaEventCreateWithFlags(&p->ev_op[i], cudaEventDisableTiming) != cudaSuccess) { set_error("plan_create: cudaEventCreate failed"); rc = ACR_B200_ECUDA; }
      if (rc == ACR_B200_OK && cudaEventCreateWithFlags(&p->ev_begin, cudaEventDisableTiming) != cudaSuccess) { set_error("plan_create: cudaEventCreate failed"); rc = ACR_B200_ECUDA; }
    }
  }
  if (rc != ACR_B200_OK) { acr_b200_plan_destroy(p); return rc; }
  *plan_out = p;
  return ACR_B200_OK;
}

extern "C" int acr_b200_plan_run(acr_b200_plan* p, const void* image, void* stream) {
  ACR_CHECK_ARG(p != nullptr, "plan_run: bad arguments");   // image may be NULL for a heads-only plan (no external op)
  cudaStream_t main_st = static_cast<cudaStream_t>(stream);
  const int n = (int)p->ops.size();
  if (p->n_streams == 1) {
    // ACR_B200_DEBUG_SYNC=1: synchronise after every launch and name the op that failed (debugging only)
    static const bool debug_sync = [] { const char* e = getenv("ACR_B200_DEBUG_SYNC"); return e && atoi(e) != 0; }();
    for (int i = 0; i < n; ++i) {
      int rc = run_one(p->ops[i], p->batch, p->arena, p->weights,
                       static_cast<const char*>(image), p->act_dtype, p->tc[i], main_st);
      if (rc) return rc;
      if (debug_sync) {
        cudaError_t e = cudaStreamSynchronize(main_st);
        if (e != cudaSuccess) {
          const acr_b200_op& o = p->ops[i];
          set_error("plan op %d failed: %s (kind %d, in C %d %dx%d stride %d, out C %d %dx%d stride %d, k %d s %d cin_pad %d cout_pad %d res %d flags %d)",
                    i, cudaGetErrorString(e), o.kind, o.in[0].C, o.in[0].H, o.in[0].W, o.in[0].pix_stride, o.out.C, o.out.H, o.out.W,
                    o.out.pix_stride, o.k, o.stride, o.cin_pad, o.cout_pad, o.has_residual, o.shift[0]);
          return ACR_B200_ECUDA;
        }
      }
    }
    return ACR_B200_OK;
  }
  // multi-stream schedule: stream 0 is the caller's stream; stream s>0 forks from it at first use and
  // every op may wait on the most recent op of other streams (wait_mask); all streams join at the end.
  int last_on[MAX_STREAMS];
  bool started[MAX_STREAMS];
  for (int s = 0; s < MAX_STREAMS; ++s) { last_on[s] = -1; started[s] = false; }
  started[0] = true;
  ACR_CHECK_CUDA(cudaEventRecord(p->ev_begin, main_st));
  for (int i = 0; i < n; ++i) {
    const acr_b200_op& op = p->ops[i];
    cudaStream_t st = op.stream_id == 0 ? main_st : p->streams[op.stream_id];
    if (!started[op.stream_id]) { ACR_CHECK_CUDA(cudaStreamWaitEvent(st, p->ev_begin, 0)); started[op.stream_id] = true; }
    for (int s = 0; s < p->n_streams; ++s)
      if ((op.wait_mask >> s) & 1) {
        if (s != op.stream_id && last_on[s] >= 0) ACR_CHECK_CUDA(cudaStreamWaitEvent(st, p->ev_op[last_on[s]], 0));
      }
    int rc = run_one(op, p->batch, p->arena, p->weights, static_cast<const char*>(image), p->act_dtype, p->tc[i], st);
    if (rc) return rc;
    ACR_CHECK_CUDA(cudaEventRecord(p->ev_op[i], st));
    last_on[op.stream_id] = i;
  }
  for (int s = 1; s < p->n_streams; ++s)
    if (last_on[s] >= 0) ACR_CHECK_CUDA(cudaStreamWaitEvent(main_st, p->ev_op[last_on[s]], 0));
  return ACR_B200_OK;
}

extern "C" int acr_b200_plan_profile(acr_b200_plan* p, const void* image, void* stream, float* ms_by_kind,
                                     int32_t* n_by_kind) {
  ACR_CHECK_ARG(p && image && ms_by_kind && n_by_kind, "plan_profile: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n = (int)p->ops.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) ACR_CHECK_CUDA(cudaEventCreate(&e));
  ACR_CHECK_CUDA(cudaEventRecord(ev[0], st));
  int rc = ACR_B200_OK;
  for (int i = 0; i < n && rc == ACR_B200_OK; ++i) {
    rc = run_one(p->ops[i], p->batch, p->arena, p->weights, static_cast<const char*>(image), p->act_dtype, p->tc[i], st);
    if (rc == ACR_B200_OK && cudaEventRecord(ev[i + 1], st) != cudaSuccess) rc = ACR_B200_ECUDA;
  }
  if (rc == ACR_B200_OK && cudaStreamSynchronize(st) != cudaSuccess) { set_error("plan_profile: sync failed: %s", cudaGetErrorString(cudaGetLastError())); rc = ACR_B200_ECUDA; }
  if (rc == ACR_B200_OK) {
    for (int k = 0; k < 16; ++k) { ms_by_kind[k] = 0.f; n_by_kind[k] = 0; }
    for (int i = 0; i < n; ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      const int k = p->ops[i].kind & 15;
      ms_by_kind[k] += ms; n_by_kind[k] += 1;
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc;
}

extern "C" int acr_b200_plan_num_launches(const acr_b200_plan* p) { return p ? (int)p->ops.size() : 0; }

extern "C" void acr_b200_plan_destroy(acr_b200_plan* p) {
  if (!p) return;
  for (ConvTcPlan* t : p->tc) conv_tc_free(t);
  for (int s = 1; s < MAX_STREAMS; ++s)
    if (p->streams[s]) cudaStreamDestroy(p->streams[s]);
  for (cudaEvent_t e : p->ev_op)
    if (e) cudaEventDestroy(e);
  if (p->ev_begin) cudaEventDestroy(p->ev_begin);
  delete p;
}

extern "C" int acr_b200_run_op(const acr_b200_op* op, int batch, void* arena, const void* weights,
                               const void* external, int act_dtype, void* stream) {
  ACR_CHECK_ARG(op && batch > 0 && arena, "run_op: bad arguments");
  return run_one(*op, batch, static_cast<char*>(arena), static_cast<const char*>(weights),
                 static_cast<const char*>(external), act_dtype, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int acr_b200_conv_describe(const acr_b200_op* op, int batch, void* arena, const void* weights,
                                      int act_dtype, int32_t* info, int n_info) {
  ACR_CHECK_ARG(op && batch > 0 && arena && weights && (info || n_info == 0), "conv_describe: bad arguments");
  ACR_CHECK_ARG(op->kind == ACR_OP_CONV && (act_dtype == ACR_DT_BF16 || act_dtype == ACR_DT_F16),
                "conv_describe: a tensor-core conv (ACR_OP_CONV, bf16 / f16) has no plan to describe otherwise");
  ConvArgs a;
  int rc = make_conv_args(*op, batch, static_cast<char*>(arena), static_cast<const char*>(weights), nullptr, &a);
  if (rc) return rc;
  ConvTcPlan* pl = nullptr;
  rc = conv_tc_prepare(a, act_dtype, &pl);
  if (rc) return rc;
  rc = conv_tc_describe(pl, info, n_info);
  conv_tc_free(pl);
  return rc;
}

// BN folding + repack, host side.  y = gamma*(conv(x)+cb-mean)/sqrt(var+eps)+beta = conv'(x) + b'
extern "C" int acr_b200_pack_conv(const float* w, const float* conv_bias, const float* g, const float* beta,
                                  const float* mean, const float* var, float eps, int cout, int cin, int k,
                                  int cout_pad, int cin_pad, int act_dtype, void* w_packed, float* bias_out) {
  ACR_CHECK_ARG(w && w_packed && bias_out && cout > 0 && cin > 0 && cout_pad >= cout && cin_pad >= cin,
                "pack_conv: bad arguments");
  ACR_CHECK_ARG(act_dtype == ACR_DT_BF16 || act_dtype == ACR_DT_F16 || act_dtype == ACR_DT_F32, "pack_conv: dtype");
  const int taps = k * k;
  for (int co = 0; co < cout_pad; ++co) {
    float scale = 1.f, shift = 0.f;
    if (co < cout) {
      if (g) { scale = g[co] / sqrtf(var[co] + eps); shift = beta[co] - mean[co] * scale; }
      if (conv_bias) shift += conv_bias[co] * scale;
    }
    bias_out[co] = co < cout ? shift : 0.f;
    for (int t = 0; t < taps; ++t)
      for (int ci = 0; ci < cin_pad; ++ci) {
        float v = 0.f;
        if (co < cout && ci < cin) v = w[((size_t)co * cin + ci) * taps + t] * scale;
        const size_t idx = ((size_t)co * taps + t) * cin_pad + ci;
        if (act_dtype == ACR_DT_BF16) static_cast<__nv_bfloat16*>(w_packed)[idx] = __float2bfloat16_rn(v);
        else if (act_dtype == ACR_DT_F16) static_cast<__half*>(w_packed)[idx] = __float2half_rn(v);
        else static_cast<float*>(w_packed)[idx] = v;
      }
  }
  return ACR_B200_OK;
}
