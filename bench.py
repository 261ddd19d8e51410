#!/usr/bin/env python
"""Benchmark of the ACR hot path (BASELINE.json metric: images/sec, 512x512, batch 256 per GPU).

    python bench.py --gpus 1 --steps 10 --warmup 3 [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU implementation (oracle port)

A "step" = one pass of the whole hot path over one batch of synthetic frames per GPU:
uint8 frames -> HRNet-W32 backbone -> heads -> centre parse -> 6D->aa -> MANO -> verts/joints
(+ one NCCL all-gather of the vertices when N > 1).  `value` times it with the frames resident
in HBM; `e2e` times the same pipeline through the public API with pinned-host frames copied H2D
and the vertices + counts read back D2H every step.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "arbitrary-hands-3d-reconstruction_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)
os.environ.setdefault("ACR_B200_SYNTHETIC_MANO", "1")

METRIC = "images/sec (512x512, HRNet-W32, two-hand MANO)"
GFLOP_PER_IMAGE = 102.12   # SURVEY.md 8d: whole network, 2*MAC (conv + linear + pooling matmuls)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def _code_digest(paths):
    """sha1 over the CODE of the given sources: // comments, blank lines and indentation do not count, so editing a
    comment does not orphan the ncu evidence that is stamped with this id."""
    import hashlib
    h = hashlib.sha1()
    for path in paths:
        with open(path) as fh:
            for line in fh:
                line = line.split("//")[0].strip()
                if line:
                    h.update(line.encode() + b"\n")
    return h.hexdigest()[:12]

def conv_build_id():
    """Digest of the conv kernel's code: ncu-derived numbers under profiles/ are stamped with it, and dropped from
    the bench line when the kernel has changed since (stale evidence must not be reported as current)."""
    return _code_digest([os.path.join(PKG, "csrc", f) for f in ("conv_tc.cu", "plan.cu")])


def load_traffic(batch):
    """(traffic_bytes, algorithmic GB, note) of the conv launch set from the newest committed ncu capture whose
    build stamp matches the current kernel; (None, None, why) otherwise."""
    import glob
    cur = conv_build_id()
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_conv_traffic.json")), reverse=True):
        try:
            with open(path) as f:
                tj = json.load(f)
        except Exception:
            continue
        if tj.get("conv_build_id") == cur and int(tj.get("batch", 256)) == batch:
            return tj["traffic_bytes"], tj["algorithmic_bytes"] / 1e9, f"ncu capture {os.path.relpath(path, ROOT)} (build {cur})"
    return None, None, f"no committed ncu capture matches the current conv build {cur} at batch {batch}"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(int(float(r[0])) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(self.rows))


def pick_threads(fn, cores):
    """Host thread count that runs `fn` -- the SAME batch that is timed afterwards -- fastest (small convs
    oversubscribe badly on 100+ cores, large batches want more threads than a single frame)."""
    import torch
    best, best_t, sweep = None, None, {}
    fn()                                    # warm caches / allocator once, not attributed to any thread count
    for n in sorted({min(cores, 64), 48, 32, 24, 16, 8}, reverse=True):   # > 64 threads: minutes per pass on these convs
        if n > cores:
            continue
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        sweep[n] = round(dt, 3)
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best, sweep


# ----------------------------------------------------------------------------- reference arm
def ref_worker(batch, steps, warmup=0, timeout=900):
    """Time the UNMODIFIED reference (snapshot oracle/_ref, made by oracle/make_ref.py from /root/reference in the
    build container; git-ignored, it travels to the GPU box with the repo) in a subprocess: the reference's
    packages are called `acr` / `mano` like our drop-in ones, so they cannot share a process with the B200 arm.
    -> dict of oracle/ref_worker.py's JSON line, or None when there is no snapshot."""
    if os.environ.get("ACR_B200_FORCE_PORT") or not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "acr")):
        return None
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_worker.py"), "--batch", str(batch), "--steps", str(steps),
                        "--warmup", str(warmup)], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        print(f"[bench] reference worker failed ({r.returncode}): {r.stderr[-400:]}", file=sys.stderr)
        return None
    j = json.loads(lines[-1])
    return None if "unavailable" in j else j


def port_pipeline(ref_batch):
    """The oracle restatement (oracle/*.py) of the same path: fall-back CPU arm when there is no snapshot."""
    import numpy as np
    import torch
    from acr_b200.synth import load_bn_calibration, make_synthetic_mano, synth_state_dict
    from oracle import mano_ref, net_ref, parse_ref
    sd = synth_state_dict(0, bn_stats=load_bn_calibration(0))
    assets = {"left": make_synthetic_mano("left"), "right": make_synthetic_mano("right")}
    gi = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (ref_batch, 512, 512, 3), generator=gi, dtype=torch.uint8)

    def step():
        out = net_ref.net_forward(sd, img)
        maps = {k: v.numpy() for k, v in out.items() if k.endswith(("_map", "_maps"))}
        p = parse_ref.parse(maps)
        L_, R_ = int(p["left_hand_num"][0]), int(p["right_hand_num"][0])
        offs = np.tile(np.array([512, 512, 0, 0, 0, 0, 0, 0, 0, 0], np.float32), (L_ + R_, 1))
        return mano_ref.mano_wrapper_forward(assets, p["params_dict"]["poses"], p["params_dict"]["betas"], L_, R_,
                                             p["params_dict"]["cam"], offs)
    return step


def cpu_arm(ref_batch, steps, warmup):
    """-> (images/s, seconds per step, cpu_baseline dict).  Thread count swept on the SAME batch that is timed."""
    cores = os.cpu_count()
    j = ref_worker(ref_batch, steps, warmup)
    if j is not None:
        dt, threads, sweep, kind, what = j["s_per_step_mean"], j["threads"], j["sweep"], "reference", j["what"]
    else:
        step = port_pipeline(ref_batch)
        threads, sweep = pick_threads(step, cores)
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = (time.perf_counter() - t0) / steps
        kind, what = "port", "oracle port (oracle/*.py; no oracle/_ref snapshot present), torch fp32 CPU"
    val = ref_batch / dt
    sample = (f"{steps} timed passes (mean) over {ref_batch} frames = a bounded sample of the batch-256 workload; {what}; "
              f"{threads} of {cores} host threads (fastest of a sweep over the same {ref_batch}-frame pass: {sweep})")
    return val, dt, {"value": val, "unit": "images/s", "cores": threads, "kind": kind, "sample": sample}


def run_reference(args):
    """The reference's own CPU implementation of the path on the host cores (all the threads that help), each step
    a bounded sample of `ref_batch` frames of the batch-256 workload.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    steps, warm = args.steps, min(args.warmup, 1)
    val, dt, cb = cpu_arm(args.ref_batch, steps, warm)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"batch {args.batch}/GPU, 512x512, HRNet-W32, two-hand MANO (BASELINE configs[2])",
                   "sample_batch": args.ref_batch},
        "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# -------------------------------------------------------------------------------- B200 arm
DUMP_BYTES = 64 << 20
# per-hand outputs of the parse kernels that fused_forward hands to its caller (top_idx / top_score / row_src are scratch)
PARSE_OUTPUTS = ("params_pred", "cam", "global_orient", "hand_pose", "betas", "poses", "detection_flag", "reorganize_idx",
                 "batch_ids", "centers_pred", "centers_conf", "hand_type", "offsets_out")


def dump_outputs(dirname, bufs, mano, max_bytes=DUMP_BYTES):
    """Write what one step returned to its caller as <dirname>/<name>.npy: the counts[2] valid rows of every parse and
    MANO output (floats as float32, integers as float64, both exact) and the row counts.  Past `max_bytes` a fixed,
    seeded subset of the rows is written; rows.npy names the rows written."""
    import numpy as np
    counts = bufs.counts.cpu().numpy()
    n = int(counts[2])
    arrays = {k: getattr(bufs, k)[:n] for k in PARSE_OUTPUTS}
    arrays.update({k: v[:n] for k, v in mano.items()})
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    arrays = {k: a.astype(np.float32 if a.dtype.kind == "f" else np.float64) for k, a in arrays.items()}
    row_bytes = 8 + sum(a.itemsize * int(np.prod(a.shape[1:])) for a in arrays.values())   # 8: the entry of rows.npy
    keep = (max_bytes - (64 << 10)) // row_bytes                                             # 64 KiB: counts + npy headers
    rows = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    arrays = {k: a[rows] for k, a in arrays.items()}
    arrays["rows"], arrays["counts"] = rows.astype(np.float64), counts.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), a)
    return arrays


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from acr.config import args as cfg_args
    from acr.main import ACR
    from acr_b200 import lib as L
    from acr_b200.synth import load_bn_calibration, make_synthetic_mano, synth_state_dict
    cfg_args().model_precision = args.dtype
    cfg_args().return_maps = False
    B = args.batch
    w48 = args.backbone == "hrnet_w48"
    if w48:     # BASELINE configs[4]'s trunk: no reference implementation exists (parity unpinned), throughput only
        from acr_b200.netspec import WIDTHS_W48, build_acr_spec
        cfg_args().hrnet_width = 48
        sd = synth_state_dict(0, spec=build_acr_spec(512, widths=WIDTHS_W48))
    else:
        sd = synth_state_dict(0, bn_stats=load_bn_calibration(0))
    assets = {"left": make_synthetic_mano("left"), "right": make_synthetic_mano("right")}
    app = ACR(state_dict=sd, mano_assets=assets)
    gi = torch.Generator().manual_seed(1000 + rank)            # every rank generates its own shard
    frames_host = torch.randint(0, 256, (B, 512, 512, 3), generator=gi, dtype=torch.uint8).pin_memory()
    frames_dev = frames_host.to(dev)
    offsets = torch.tensor([[512., 512, 0, 0, 0, 0, 0, 0, 0, 0]], device=dev).repeat(B, 1)
    from acr_b200.dist import PeerVertexGather, gather_vertices
    gather_buf = gather_cnt = peers = None
    gather_mode = "single GPU"
    if world > 1:
        gather_cnt = torch.empty(world, 8, dtype=torch.int32, device=dev)
        if args.gather == "fused":
            try:   # vertex all-gather fused into the MANO kernel (multimem.st / peer stores over NVLink)
                peers = PeerVertexGather(2 * B, dev)
                gather_mode = (f"vertex + count all-gather fused into mano_forward_kernel: {peers.mode} over NVLink into "
                               "double-buffered slots, arrival flags (no barrier, no NCCL call)")
            except Exception as e:  # noqa: BLE001
                if rank == 0:
                    print(f"[bench] symmetric memory unavailable ({e!r}); using the NCCL all-gather", file=sys.stderr)
        if peers is None:
            gather_buf = torch.empty(world, 2 * B, 778, 3, device=dev)
            gather_mode = "1 NCCL all-gather of the vertices"
    # the FULL result of a step goes back to the host in the e2e path: vertices, joints, MANO parameters, counts
    R2 = 2 * B
    host = {"verts": torch.empty(R2, 778, 3).pin_memory(), "joints": torch.empty(R2, 21, 3).pin_memory(),
            "poses": torch.empty(R2, 48).pin_memory(), "betas": torch.empty(R2, 10).pin_memory(),
            "cam": torch.empty(R2, 3).pin_memory(), "counts": torch.empty(8, dtype=torch.int32).pin_memory()}

    def step(frames):
        """One pass of the hot path.  With N > 1 the one exchange of the path -- every shard's vertices (and row
        counts) on every rank -- happens inside the MANO kernel (fused mode: stores over NVLink, no barrier, no
        NCCL call; arrival of step k is awaited when it is consumed / at the end of the timed region) or as one
        NCCL all-gather right after it (--gather nccl)."""
        bufs, mano = app.fused_forward(frames, offsets, peers=peers)
        if world > 1 and peers is None:
            gather_vertices(mano["verts"], bufs.counts, gather_buf, gather_cnt)
        return bufs, mano

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, n):
        """n calls between CUDA events, barrier + synchronize on both sides, MAX over ranks.  In fused-gather mode the
        arrival of the LAST step's data from every rank is awaited inside the timed region."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        for _ in range(n):
            fn()
        if peers is not None:
            peers.finish()
        e1.record()
        sync_all()
        mine = e0.elapsed_time(e1)
        ms = torch.tensor([mine], device=dev)
        per_rank = [mine]
        if world > 1:
            allms = [torch.zeros(1, device=dev) for _ in range(world)]
            dist.all_gather(allms, ms)
            per_rank = [float(t.item()) for t in allms]
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), per_rank

    warm = max(3, args.warmup)             # timing rule: at least 3 untimed steps before the timed region
    for _ in range(warm):
        step(frames_dev)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    last = {}

    def value_step():
        last["out"] = step(frames_dev)

    ms_value, ms_per_rank = timed(value_step, args.steps)
    if args.dump_outputs and rank == 0:        # before any later call re-uses the parse buffers
        dump_outputs(args.dump_outputs, *last["out"])

    # ---- end to end: every step copies ITS frames from pinned host memory and reads ITS results back.
    # Two device staging buffers + a copy stream let the H2D of step i+1 overlap the kernels of step i
    # (the copy engine is idle otherwise); the result read-back of step i is awaited before step i+1 ends.
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [torch.empty_like(frames_dev) for _ in range(2)]
    staged = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"i": 0, "primed": False}

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])          # the kernels that read this slot are done
            stage[slot].copy_(frames_host, non_blocking=True)
            staged[slot].record(copy_stream)

    def e2e_step():
        cur = torch.cuda.current_stream()
        i = state["i"]
        if not state["primed"]:
            for sl in range(2):
                consumed[sl].record(cur)
            prefetch(i & 1)
            state["primed"] = True
        prefetch((i + 1) & 1)                                 # next step's frames, overlapped
        cur.wait_event(staged[i & 1])
        bufs, mano = step(stage[i & 1])
        consumed[i & 1].record(cur)
        host["verts"].copy_(mano["verts"], non_blocking=True)
        host["joints"].copy_(mano["joints"], non_blocking=True)
        host["poses"].copy_(bufs.poses, non_blocking=True)
        host["betas"].copy_(bufs.betas, non_blocking=True)
        host["cam"].copy_(bufs.cam, non_blocking=True)
        host["counts"].copy_(bufs.counts, non_blocking=True)
        cur.synchronize()                                     # the caller consumes the result every step
        state["i"] = i + 1

    for _ in range(3):
        e2e_step()
    ms_e2e, _ = timed(e2e_step, args.steps)
    clocks = sampler.stop() if sampler else None

    # ---- N > 1: verify the exchange OUTSIDE the timed region -- every shard of the gathered buffer (fused mode: the
    # slot written by the MANO kernels of all ranks; nccl mode: the collective's output) against an independent NCCL
    # all-gather of the same step's local vertices and counts, on every rank
    gather_check = None
    if world > 1:
        bufs, mano = step(frames_dev)
        if peers is not None:
            peers.finish()
            got_v, got_c = peers.gathered(), peers.counts()
        else:
            got_v, got_c = gather_buf, gather_cnt
        ref_v = torch.empty(world, 2 * B, 778, 3, device=dev)
        ref_c = torch.empty(world, 8, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(ref_v.view(-1), mano["verts"].contiguous().view(-1))
        dist.all_gather_into_tensor(ref_c.view(-1), bufs.counts)
        torch.cuda.synchronize()
        ok = bool(torch.equal(got_c, ref_c))
        for r in range(world):
            nv = int(ref_c[r, 2])
            ok = ok and nv > 0 and bool(torch.equal(got_v[r, :nv], ref_v[r, :nv]))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_check = bool(flag.item())

    # ---- MANO kernel alone (BASELINE metric, second half): CUDA events around the kernel at the step's own size
    # (2B rows, L2 flushed between launches) and at 65 536 hands (outputs 1.3 GB >> L2); vertices vs the oracle
    from acr_b200 import ops as _ops
    ml_, mr_ = app.mano_regression.models()

    def mano_alone(n, iters, flush):
        g = torch.Generator().manual_seed(5)
        poses = (torch.randn(n, 48, generator=g) * 0.5).to(dev)
        betas_ = torch.randn(n, 10, generator=g).to(dev)
        cam_ = (torch.rand(n, 3, generator=g) + 0.5).to(dev)
        offs_ = offsets[:1].repeat(n, 1)
        ht_ = (torch.arange(n, device=dev) >= n // 2).int()
        scratch = torch.empty(64 << 20, dtype=torch.float32, device=dev) if flush else None   # 256 MB > 126 MB L2
        for _ in range(3):
            out = _ops.mano_forward(ml_, mr_, poses, betas_, ht_, 1, 9, cam_, offs_)
        tot = 0.0
        for _ in range(iters):
            if flush:
                scratch.fill_(1.0)
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            out = _ops.mano_forward(ml_, mr_, poses, betas_, ht_, 1, 9, cam_, offs_)
            eb.record()
            torch.cuda.synchronize()
            tot += ea.elapsed_time(eb)
        return tot / iters * 1e3, (poses, betas_, cam_, offs_, ht_, out)      # us per launch

    mano_small_us, mano_io = mano_alone(2 * B, 10, True)
    mano_big_us, _ = mano_alone(65536, 5, False)

    # ---- roofline of the dominant kernel (the tcgen05 conv), measured live with CUDA events
    eng = app.model.engine(B, dev)
    eng.profile(frames_dev)
    prof = [eng.profile(frames_dev) for _ in range(2)][-1]
    conv_ms, conv_n = prof.get(L.OP_CONV, (0.0, 0))
    total_prof_ms = sum(v[0] for v in prof.values())
    bufs, mano = step(frames_dev)
    torch.cuda.synchronize()
    n_hands = int(bufs.counts[2])
    if rank == 0:
        peaks = load_peaks()
        traffic, alg_gb, traffic_note = (None, None, "no ncu capture of the W48 plan") if w48 else load_traffic(B)
        # MANO vertices of the stand-alone launch above vs the oracle (numpy restatement pinned to the reference)
        from oracle import mano_ref as _mano_ref
        poses_, betas_, cam_, offs_, ht_, mo = mano_io
        nchk = min(64, poses_.shape[0])
        idx = torch.cat([torch.arange(nchk // 2), torch.arange(poses_.shape[0] - nchk // 2, poses_.shape[0])])
        Lc = int((ht_[idx] == 0).sum())
        assets_np = {"left": assets["left"], "right": assets["right"]}
        mref = _mano_ref.mano_wrapper_forward(assets_np, poses_[idx].cpu().numpy(), betas_[idx].cpu().numpy(), Lc, nchk - Lc,
                                              cam_[idx].cpu().numpy(), offs_[idx].cpu().numpy())
        verts_err = float(np.abs(mo["verts"][idx].cpu().numpy() - mref["verts"]).max())
        verts_rel = float(verts_err / np.abs(mref["verts"]).max())
        MANO_BYTES = 19324        # SURVEY.md 8d: 232 B in + verts 9 336 + joints 252 (+ verts_camed 9 336 + pj2d 168)
        MANO_FLOP = 1.152e6
        mano_gbs = lambda n, us: n * MANO_BYTES / us / 1e3
        conv_gflop = sum(2.0 * o.out.H * o.out.W * o.out.C * o.ins[0].C * o.attrs["k"] ** 2
                         for o in eng.spec.ops if o.kind == "conv") / 1e9
        if any(r["kind"] == L.OP_IM2COL_STEM for r in eng.recs):   # ACR_B200_STEM_FUSED=0: conv1 (3x3 s2, 3 -> 64) as im2col + a
            # 1x1 conv_tc launch (27 real taps) is part of the conv launch set; the fused stem_tc_kernel (default) is timed and
            # counted apart (profile_ms_by_kind["11"]), so neither its time nor its flops enter this roofline
            conv_gflop += sum(2.0 * o.out.H * o.out.W * 64 * 27 for o in eng.spec.ops if o.kind == "stem") / 1e9
        ach = conv_gflop * B / conv_ms if conv_ms else 0.0          # TFLOP/s (GFLOP/ms)
        img_s = world * B * args.steps / (ms_value / 1e3)
        e2e_s = world * B * args.steps / (ms_e2e / 1e3)
        launches = eng.num_launches + 3 + 1 + (1 if cfg_args().cam_trans_mode == "lstsq" else 0)
        out = {
            "metric": METRIC.replace("W32", "W48") if w48 else METRIC, "value": img_s, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_value / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": (f"batch {B}/GPU, 512x512 uint8 RGB, HRNet-W48 trunk (restated: the reference ships only W32 -- PARITY "
                                    "UNPINNED, throughput only), two-hand MANO (BASELINE configs[4] per GPU)") if w48 else
                                   f"batch {B}/GPU, 512x512 uint8 RGB, HRNet-W32, two-hand MANO (BASELINE configs[2])",
                       "global_batch": B * world, "hands_per_step_rank0": n_hands,
                       "parallelism": f"frames sharded over {world} rank(s); {gather_mode}" if world > 1 else "single GPU",
                       "l2_hygiene": f"inputs {B * 786432 / 2**20:.0f} MiB + {eng.arena_bytes / 2**20:.0f} MiB activations per step >> 126 MB L2",
                       "weights": "seeded synthetic (no checkpoint ships with the reference)"},
            "clocks": clocks,
            "e2e": {"value": e2e_s, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(frames_host.numel()),
                    "d2h_bytes_per_step": int(sum(t.numel() * t.element_size() for t in host.values())),
                    "d2h_contents": "verts, joints, poses, betas, cam of the worst-case 2B rows + row counts"},
            "gpu_launches": launches * args.steps,
            "roofline": {"kernel": f"conv_tc_kernel (tcgen05 implicit-GEMM conv, all {conv_n} launches of a step)",
                         "bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": ach / peaks["tf_sustained"] if ach else 0.0, "traffic": traffic,
                         "traffic_note": "DRAM read+write bytes of the whole conv launch set per step: " + traffic_note
                                         + (f" (algorithmic: {alg_gb:.1f} GB)" if alg_gb else ""),
                         "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                         "algorithmic_gflop_per_launch_set": conv_gflop * B,
                         "conv_ms_per_step": conv_ms, "conv_share_of_plan": conv_ms / total_prof_ms if total_prof_ms else None,
                         "whole_net_tflops": eng.flops_per_image / 1e9 * B / (ms_value / args.steps)},
            "profile_ms_by_kind": {str(k): round(v[0], 3) for k, v in prof.items()},
            # BASELINE metric, second half + north-star MANO target (>= 0.60 of the HBM roofline): the kernel alone
            "mano_verts_max_abs_err": verts_err,
            "mano_verts_max_rel_err": verts_rel,
            "roofline_mano": {"kernel": "mano_forward_kernel", "bound": "hbm", "unit": "GB/s", "peak": peaks["hbm_gbs"],
                              "peak_source": peaks["source"], "bytes_per_hand": MANO_BYTES, "flop_per_hand": MANO_FLOP,
                              "achieved": mano_gbs(2 * B, mano_small_us), "frac": mano_gbs(2 * B, mano_small_us) / peaks["hbm_gbs"],
                              "hands": 2 * B, "us_per_launch": mano_small_us, "l2": "flushed between launches",
                              "at_65536_hands": {"us_per_launch": mano_big_us, "achieved": mano_gbs(65536, mano_big_us),
                                                 "frac": mano_gbs(65536, mano_big_us) / peaks["hbm_gbs"],
                                                 "fp32_tflops": 65536 * MANO_FLOP / mano_big_us / 1e6},
                              "note": "1.15 MFLOP of fp32 FMA per 19.3 KB hand: the kernel is FP32-issue bound (FFMA2), not HBM bound"},
        }
        if world > 1:
            out["gather_check"] = gather_check
            out["ms_per_step_by_rank"] = [round(m / args.steps, 3) for m in ms_per_rank]
        if args.cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(args):
    """The reference's CPU path timed on the host cores, bounded sample (rank 0, N=1 only)."""
    return cpu_arm(args.ref_batch, 2, 0)[2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--backbone", default="hrnet_w32", choices=["hrnet_w32", "hrnet_w48"],
                    help="hrnet_w48: the wider trunk of BASELINE configs[4]; no reference exists for it (parity unpinned)")
    ap.add_argument("--ref-batch", type=int, default=8, help="frames per CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="N>1: vertex all-gather fused into the MANO kernel (symmetric memory) or a separate NCCL call")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    if args.gpus > 1 or args.backbone != "hrnet_w32":
        args.cpu_baseline = False          # the CPU arm is the reference's own network (HRNet-W32)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
