"""Many video streams per batch on the GPU: per-frame parse (acr_b200_parse_per_frame), per-stream OneEuro state
(acr_b200_one_euro_smooth_streams) and ACR.stream_forward / capture_graph(streams=), against the reference-pinned
oracles of tests/stream_oracle.py and against the single-stream path."""
import os

import numpy as np
import pytest
import torch

from tests import stream_oracle as so
from tests.helpers import GOLDEN
from tests.test_oracle_golden import make_parse_case

pytestmark = pytest.mark.gpu

ROW_KEYS = ("params_pred", "cam", "global_orient", "hand_pose", "betas", "poses", "detection_flag", "reorganize_idx",
            "batch_ids", "centers_pred", "centers_conf", "hand_type", "offsets_out")


def _parse(maps_np, meta_ids=None, offsets=None, per_frame=True):
    """Both parse exports on NCHW numpy maps uploaded as NHWC (like test_gpu_parse.py) -> dict of numpy arrays:
    every row buffer (all 2B rows) and counts[:6]."""
    from acr_b200 import ops
    B = maps_np["l_center_map"].shape[0]
    names = dict(l_center="l_center_map", r_center="r_center_map", l_params="l_params_maps",
                 r_params="r_params_maps", l_prior="l_prior_maps", r_prior="r_prior_maps")
    maps = {}
    for k, n in names.items():
        t = torch.from_numpy(maps_np[n]).cuda().permute(0, 2, 3, 1).contiguous()
        maps[k] = (t, t.shape[-1])
    bufs = ops.ParseBuffers(B, "cuda")
    ids = None if meta_ids is None else torch.as_tensor(meta_ids, dtype=torch.int64).cuda()
    offs = None if offsets is None else torch.as_tensor(offsets).float().cuda()
    ops.parse_maps(maps, B, bufs, ids, offs, 0.35, per_frame=per_frame)
    torch.cuda.synchronize()
    out = {k: getattr(bufs, k).cpu().numpy() for k in ROW_KEYS}
    out["counts"] = bufs.counts[:6].cpu().numpy()
    return out


def _equal(a, b, rows_a=None, rows_b=None, skip=()):
    for k in ROW_KEYS + ("counts",):
        if k in skip:
            continue
        x = a[k] if rows_a is None or k == "counts" else a[k][rows_a]
        y = b[k] if rows_b is None or k == "counts" else b[k][rows_b]
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)), k   # bit for bit


@pytest.mark.parametrize("t", range(so.T))
def test_parse_per_frame_golden(t):
    """acr_b200_parse_per_frame on the golden's maps vs the reference's batch-of-one parse of every frame."""
    g = np.load(os.path.join(GOLDEN, "stream_golden.npz"))
    out = _parse(so.make_stream_maps(t), so.stream_meta_ids(t))
    for k, ref in (("detection_flag", g["detection_flag"][t]), ("reorganize_idx", g["reorganize_idx"][t]),
                   ("centers_pred", g["centers_pred"][t]), ("counts", g["counts"][t])):
        assert out[k].shape == ref.shape and (out[k] == ref).all(), k
    assert (out["hand_type"] == np.repeat([0, 1], so.S)).all()
    assert (out["batch_ids"] == np.tile(np.arange(so.S), 2)).all()
    for k in ("params_pred", "centers_conf"):
        assert np.abs(out[k] - g[k][t]).max() < 1e-6, k
    for k in ("cam", "global_orient", "hand_pose", "betas", "poses"):
        assert np.abs(out[k] - g[k][t]).max() < 5e-5, k


@pytest.mark.parametrize("case", ["both", "no_left", "mixed", "none", "far"])
def test_per_frame_equals_batch_parse_at_batch_one(case):
    """At B = 1 the per-frame parse IS the reference's parse: bit for bit equal to acr_b200_parse, on every frame of
    every parse_golden case cut to a batch of one."""
    g = np.load(os.path.join(GOLDEN, "parse_golden.npz"))
    maps = make_parse_case(case, int(g[f"{case}__B"]))
    for b in range(maps["l_center_map"].shape[0]):
        one = {k: np.ascontiguousarray(v[b:b + 1]) for k, v in maps.items()}
        offs = np.arange(10, dtype=np.float32)[None] + b
        _equal(_parse(one, [7 + b], offs, per_frame=True), _parse(one, [7 + b], offs, per_frame=False))


def _random_maps(B, seed):
    g = np.random.default_rng(seed)
    maps = {}
    for s in "lr":
        cm = (g.standard_normal((B, 1, 64, 64), dtype=np.float32) * 0.05)
        on = g.random(B) > 0.3                         # ~30 % of the centres removed
        on[1:3] = False                                # frames 1 and 2 without any hand
        if s == "l":
            on[0] = False                              # frame 0 without its left hand
        for b in np.nonzero(on)[0]:
            cm[b, 0, g.integers(0, 64), g.integers(0, 64)] = 0.5 + g.random()
        maps[f"{s}_center_map"] = cm
        maps[f"{s}_params_maps"] = g.standard_normal((B, 109, 64, 64), dtype=np.float32)
        maps[f"{s}_prior_maps"] = g.standard_normal((B, 106, 64, 64), dtype=np.float32) * 0.1
    return maps


def test_batch_independence():
    """B = 64 frames: each slot's two rows equal a B = 1 launch on that frame alone, bit for bit; permuting the
    frames permutes the rows and nothing else."""
    B = 64
    maps = _random_maps(B, 11)
    meta = np.arange(B) * 3 + 1
    offs = np.random.default_rng(12).standard_normal((B, 10)).astype(np.float32)
    full = _parse(maps, meta, offs)
    assert (full["counts"][:3] == [B, B, 2 * B]).all()
    assert 0 < full["counts"][4] < B - 3 and 0 < full["counts"][5] < B - 2
    assert (full["detection_flag"][[1, 2, B + 1, B + 2]] == 0).all()
    for b in range(B):
        one = _parse({k: np.ascontiguousarray(v[b:b + 1]) for k, v in maps.items()}, meta[b:b + 1], offs[b:b + 1])
        _equal(full, one, rows_a=[b, B + b], rows_b=[0, 1], skip=("batch_ids", "counts"))
        assert (full["batch_ids"][[b, B + b]] == b).all()
    perm = np.random.default_rng(13).permutation(B)
    pm = _parse({k: np.ascontiguousarray(v[perm]) for k, v in maps.items()}, meta[perm], offs[perm])
    rows = np.concatenate([perm, B + perm])
    _equal(pm, full, rows_b=rows, skip=("batch_ids",))
    assert (pm["batch_ids"] == np.tile(np.arange(B), 2)).all()


def test_streams_vs_oracle():
    """40 streams over 12 steps, 16 slots a step: a random subset of the streams in random order, -1 padding slots,
    random detection dropouts and resets between steps, against one OneEuroBank pair per stream.  Padding slots
    and out-of-range ids filter nothing and leave every state byte of the streams not in the batch unchanged."""
    from acr_b200 import ops
    NS, T, B = 40, 12, 16
    g = np.random.default_rng(5)
    states = ops.StreamStates(NS, "cuda")
    sm = so.StreamSmoother(4.0)
    ht = torch.tensor(np.repeat([0, 1], B), dtype=torch.int32).cuda()
    bi = torch.tensor(np.tile(np.arange(B), 2), dtype=torch.int64).cuda()
    base = (g.standard_normal((NS, 2, 48)) * 0.5).astype(np.float32)
    checked = 0
    for t in range(T):
        if t in (4, 8):
            rs = g.choice(NS, 5, replace=False)
            states.reset(rs)
            for s in rs:
                sm.reset(s)
        n_live = 10 if t == 6 else int(g.integers(8, B + 1))
        ids = np.full(B, -1, np.int32)
        ids[g.choice(B, n_live, replace=False)] = g.choice(NS, n_live, replace=False)
        oracle_ids = ids.copy()
        dev_ids = None
        if t == 6:       # ids the host check rejects reach the kernel only from the device: they are padding too
            ids[np.nonzero(ids < 0)[0][:3]] = [NS, 1000, -5]
            dev_ids = torch.from_numpy(ids).cuda()
        poses = base[np.clip(ids, 0, NS - 1)].transpose(1, 0, 2).reshape(2 * B, 48) + \
            (g.standard_normal((2 * B, 48)) * 0.2).astype(np.float32)
        betas = (g.standard_normal((2 * B, 10)) * 0.3).astype(np.float32)
        det = (g.random(2 * B) > 0.2).astype(np.float32)
        st0 = states.state.view(NS, -1).clone()
        p, b_ = torch.from_numpy(poses).cuda(), torch.from_numpy(betas).cuda()
        ops.one_euro_smooth_streams(p, b_, states, dev_ids if dev_ids is not None else ids, hand_type=ht,
                                    detection_flag=torch.from_numpy(det).cuda(), batch_ids=bi, smooth_coeff=4.0)
        rp, rb = sm.apply(poses, betas, ht.cpu().numpy(), det, bi.cpu().numpy(), oracle_ids)
        gp, gb = p.cpu().numpy(), b_.cpu().numpy()
        assert np.abs(gp - rp).max() < 5e-5, t
        assert np.abs(gb - rb).max() < 1e-6, t
        skipped = (det == 0) | (np.tile(oracle_ids, 2) < 0)
        assert np.array_equal(gp[skipped], poses[skipped]) and np.array_equal(gb[skipped], betas[skipped])
        checked += int((~skipped).sum())
        live = set(int(s) for s in oracle_ids if s >= 0)
        untouched = [s for s in range(NS) if s not in live]
        assert torch.equal(states.state.view(NS, -1)[untouched].view(torch.int32), st0[untouched].view(torch.int32)), t
    assert checked > 150


def test_stream_ids_host_validation():
    from acr_b200 import ops
    states = ops.StreamStates(4, "cuda")
    p, b = torch.zeros(4, 48).cuda(), torch.zeros(4, 10).cuda()
    kw = dict(hand_type=torch.tensor([0, 0, 1, 1], dtype=torch.int32).cuda(), detection_flag=None,
              batch_ids=torch.tensor([0, 1, 0, 1]).cuda())
    for bad in ([1, 1], [0, 4], [0.0, 1.0], [[0, 1]]):
        with pytest.raises((ValueError, TypeError)):
            ops.one_euro_smooth_streams(p, b, states, bad, **kw)
    ops.one_euro_smooth_streams(p, b, states, [-1, 3], **kw)
    torch.cuda.synchronize()
    blocks = states.state.view(4, -1)
    assert (blocks[:3] == 0).all() and (blocks[3] != 0).any()
    states.reset([3])
    assert (states.state == 0).all()


# ------------------------------------------------------------------------------------------ whole pipeline
@pytest.fixture(scope="module")
def app_parts():
    os.environ.setdefault("ACR_B200_SYNTHETIC_MANO", "1")
    from acr_b200.synth import load_bn_calibration, make_synthetic_mano, synth_state_dict
    sd = synth_state_dict(0, bn_stats=load_bn_calibration(0))
    assets = {"left": make_synthetic_mano("left"), "right": make_synthetic_mano("right")}
    gi = torch.Generator().manual_seed(123)
    img = torch.randint(0, 256, (2, 512, 512, 3), generator=gi, dtype=torch.uint8)
    return sd, assets, img


def _frames(img, B, step):
    """B frames of step `step`: the two seed-123 test frames, slightly perturbed per step and slot."""
    g = torch.Generator().manual_seed(1000 + step)
    noise = torch.randint(-6, 7, (B, 512, 512, 3), generator=g, dtype=torch.int16)
    return (img[torch.arange(B) % 2].to(torch.int16) + noise).clamp(0, 255).to(torch.uint8)


MANO_KEYS = ("verts", "joints", "center", "verts_camed", "pj2d", "pj2d_org", "cam_trans")


def _snapshot(bufs, mano):
    out = {k: getattr(bufs, k).clone() for k in ROW_KEYS}
    out["counts"] = bufs.counts.clone()
    out.update({"mano_" + k: mano[k].clone() for k in MANO_KEYS if k in mano})
    return out


def test_graph_equals_eager(app_parts):
    """capture_graph(4, streams=) replayed for 6 steps with changing stream ids (padding included, a reset in
    between) equals eager stream_forward on its own StreamStates, bit for bit: parse buffers, MANO outputs, state."""
    from acr.main import ACR
    from acr_b200 import ops
    sd, assets, img = app_parts
    app = ACR(state_dict=sd, mano_assets=assets)
    B, NS = 4, 8
    st_graph, st_eager = ops.StreamStates(NS, "cuda"), ops.StreamStates(NS, "cuda")
    replay = app.capture_graph(B, streams=st_graph)
    assert (st_graph.state == 0).all()             # capturing filtered nothing
    offs = torch.tensor([[512., 512, 0, 0, 0, 0, 0, 0, 0, 0]]).repeat(B, 1).cuda()
    schedule = [None, [3, 0, 5, 1], [3, -1, 5, 7], [6, 2, -1, -1], [3, 0, 5, 1], [1, 3, 0, 5]]
    n_det = 0
    for step, ids in enumerate(schedule):
        if step == 4:
            st_graph.reset([3]); st_eager.reset([3])
        frames = _frames(img, B, step).cuda()
        e = _snapshot(*app.stream_forward(frames, offs, st_eager, ids))
        gr = _snapshot(*replay(frames, offs, ids))
        torch.cuda.synchronize()
        for k in e:
            assert torch.equal(e[k], gr[k]), (step, k)
        n_det += int(e["counts"][3])
    assert torch.equal(st_graph.state.view(torch.int32), st_eager.state.view(torch.int32))
    print(f"graph == eager over {len(schedule)} steps, {n_det} detected hands")


def test_stream_forward_matches_single_stream_path(app_parts):
    """Two streams through stream_forward at B = 2 over 4 steps == each stream through its own ACR.batch_forward at
    B = 1 with temporal_optimization: params, smoothed poses, verts and joints bit for bit."""
    from acr.main import ACR
    from acr_b200 import ops
    sd, assets, img = app_parts
    app = ACR(state_dict=sd, mano_assets=assets)
    app.temporal_optimization = True
    singles = []
    for _ in range(2):
        a = ACR(state_dict=sd, mano_assets=assets)
        a.temporal_optimization = True
        singles.append(a)
    states = ops.StreamStates(2, "cuda")
    offs = torch.tensor([[512., 512, 0, 0, 0, 0, 0, 0, 0, 0]]).repeat(2, 1)
    n_det = 0
    for step in range(4):
        frames = _frames(img, 2, 100 + step)
        bufs, mano = app.stream_forward(frames.cuda(), offs.cuda(), states)
        got = {"params_pred": bufs.params_pred, "poses": bufs.poses, "betas": bufs.betas, "verts": mano["verts"],
               "j3d": mano["joints"], "detection_flag": bufs.detection_flag}
        got = {k: v.clone() for k, v in got.items()}
        for s in range(2):
            ref = singles[s].batch_forward(frames[s:s + 1].cuda())
            want = {"params_pred": ref["params_pred"], "poses": ref["params_dict"]["poses"],
                    "betas": ref["params_dict"]["betas"], "verts": ref["verts"], "j3d": ref["j3d"],
                    "detection_flag": ref["detection_flag"]}
            for k, w in want.items():
                assert torch.equal(got[k][[s, 2 + s]], w), (step, s, k)
            n_det += int(ref["detection_flag"].sum())
    print(f"stream_forward == single-stream batch_forward over 4 steps, {n_det} detected hands")
