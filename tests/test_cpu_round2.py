"""CPU tests of the round-2 host logic: fp32 / heads-only plan layouts, the same-rounding oracle and the per-op
oracle against the whole-network oracle, the reference snapshot, the gather layout / C struct, bench helpers and
the stale-output guard."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def sd():
    from acr_b200.synth import load_bn_calibration, synth_state_dict
    return synth_state_dict(0, bn_stats=load_bn_calibration(0))


@pytest.fixture(scope="module")
def image():
    gi = torch.Generator().manual_seed(123)
    return torch.randint(0, 256, (1, 512, 512, 3), generator=gi, dtype=torch.uint8)


def test_fp32_and_heads_only_plan_layouts():
    from acr_b200 import lib as L
    from acr_b200.engine import Engine
    full16 = Engine(None, 2, "cpu", torch.bfloat16, dry_run=True)
    full32 = Engine(None, 2, "cpu", torch.float32, dry_run=True)
    heads = Engine(None, 2, "cpu", torch.bfloat16, dry_run=True, head_only=True)
    # fp32 plan: CUDA-core stem where the 16-bit plan has the fused tcgen05 stem, every conv on the validation kernel
    assert full32.n_ops == full16.n_ops
    assert all(r["kind"] not in (L.OP_CONV, L.OP_IM2COL_STEM, L.OP_STEM_TC) for r in full32.recs)
    assert 1.9 < full32.arena_bytes / full16.arena_bytes < 2.1
    # heads-only plan = the ops from the coord concat on; the external feature buffer is allocated up front
    first = next(i for i, r in enumerate(full16.recs) if r["kind"] == L.OP_COORD)
    assert heads.n_ops == full16.n_ops - first == 53
    assert heads.recs[0]["kind"] == L.OP_COORD
    xcat = heads.spec.tensors["feat32"].base.name
    assert heads.geo[xcat]["offset"] is not None


def test_same_rounding_oracle_and_head_forward(sd, image):
    from oracle import net_ref
    a = net_ref.net_forward(sd, image, return_backbone=True)
    b = net_ref.net_forward(sd, image, torch.float16, fold_round=True)
    rel = lambda x, y: float((x - y).abs().max() / y.abs().max())
    for k in ("segms", "l_center_map", "r_params_maps", "pooled"):
        e = rel(b[k], a[k])
        assert 1e-5 < e < 0.08, (k, e)          # rounded storage moves the result, but only by storage round-off
    with pytest.raises(AssertionError):
        net_ref._Net(sd, None, fold_round=True)
    h = net_ref.head_forward(sd, a["backbone"])
    for k in ("segms", "l_center_map", "l_params_maps", "r_prior_maps"):
        assert torch.equal(h[k], a[k]), k


def test_op_oracle_matches_network_oracle(sd, image):
    """The per-op restatement (teacher-forced sweep) is the same arithmetic as the whole-network oracle."""
    from oracle import net_ref, op_ref
    sdf = {k: v.float() for k, v in sd.items() if v.dtype.is_floating_point}
    n = net_ref._Net(sd)
    x = (image.float().permute(0, 3, 1, 2) / 255.0) * 2.0 - 1.0
    s1 = n.cbr(x, "backbone.conv1", "backbone.bn1", stride=2)
    assert torch.allclose(op_ref.stem(image, sdf), s1, atol=1e-6)
    assert torch.allclose(op_ref.stem_from_cols(op_ref.im2col_stem(image), sdf), s1, atol=2e-5)
    s2 = op_ref.conv_bn_act(s1, sdf, "backbone.conv2", "backbone.bn2", 2, True)
    assert torch.allclose(s2, n.cbr(s1, "backbone.conv2", "backbone.bn2", stride=2), atol=1e-6)
    y = op_ref.conv_bn_act(s2, sdf, "backbone.layer1.0.conv1", "backbone.layer1.0.bn1", 1, True)
    assert y.shape == (1, 64, 128, 128)
    t = [torch.randn(1, 8, 16, 16), torch.randn(1, 8, 8, 8), torch.randn(1, 8, 4, 4)]
    exp = torch.relu(t[0] + torch.nn.functional.interpolate(t[1], scale_factor=2) + torch.nn.functional.interpolate(t[2], scale_factor=4))
    assert torch.equal(op_ref.fuse(t, [0, 1, 2]), exp)
    c = op_ref.coord(128, 128)
    assert c[0, 5, 0] == -1 and c[0, 5, 127] == 1 and c[1, 0, 7] == -1 and c[1, 127, 7] == 1
    # part branch: pool -> offsets -> final conv == the network oracle's params maps
    full = net_ref.net_forward(sd, image, return_backbone=True)
    nn_ = net_ref._Net(sd)
    xb = full["backbone"]
    lin = torch.arange(128, dtype=torch.float32) / 127 * 2 - 1
    xc = torch.cat([xb, torch.stack([lin.view(1, 128).expand(128, 128), lin.view(128, 1).expand(128, 128)])[None]], 1)
    contact = nn_.cbr(xc, "contact_layers.1.0", "contact_layers.1.1")
    pooled = op_ref.attention_pool(contact, full["segms"])
    assert torch.allclose(pooled, full["pooled"], atol=1e-5)
    for s in "lr":
        prm = nn_.head_stack(xc, f"{s}_final_layers.1")
        cam = nn_.head_stack(xc, f"{s}_final_layers.3")
        cam = torch.cat([torch.pow(1.1, cam[:, :1]), cam[:, 1:]], 1)
        out = op_ref.final_params(prm, cam, op_ref.part_offsets(pooled, sdf, s), sdf, s)
        assert float((out - full[f"{s}_params_maps"]).abs().max()) < 1e-4 * float(full[f"{s}_params_maps"].abs().max())


def test_reference_snapshot_reproduces_the_golden():
    """oracle/_ref (made by oracle/make_ref.py, git-ignored) is what the reference arm of bench.py times: when it is
    present it must BE the reference, i.e. reproduce tests/golden/net_golden.npz exactly."""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "acr")):
        pytest.skip("no oracle/_ref snapshot in this checkout (made by __graft_entry__.build() where /root/reference exists)")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_worker.py"), "--check"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    j = json.loads(line)
    assert r.returncode == 0 and j["same_centres"] and j["verts_rel_err"] < 1e-6, (r.returncode, line, r.stderr[-500:])


def test_gather_layout_and_c_struct():
    from acr_b200 import lib as L
    from acr_b200.dist import gather_layout
    assert C.sizeof(L.Gather) == 8 * 8 + 8 + 4 + 4 + 8 + 8 + 8 + 8 + 8          # acr_b200_gather, include/acr_b200.h
    for world, rows in ((2, 64), (4, 512), (8, 512), (8, 2)):
        lay = gather_layout(world, rows)
        assert lay["counts_offset"] % 16 == 0 and lay["slot_bytes"] % 16 == 0 and lay["flags_offset"] % 16 == 0
        assert lay["counts_offset"] >= world * rows * 778 * 3 * 4
        assert lay["slot_bytes"] >= lay["counts_offset"] + world * 32
        assert lay["flags_offset"] == 2 * lay["slot_bytes"] and lay["total_bytes"] >= lay["flags_offset"] + world * 8
        # every rank's row block starts on a 16-byte boundary shared with the local layout (rows even => (r*rows*2334) % 4 == 0)
        for r in range(world):
            assert (r * rows * 778 * 3) % 4 == 0
    with pytest.raises(ValueError):
        gather_layout(2, 63)


def test_bench_traffic_stamp_and_thread_sweep(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    bid = bench.conv_build_id()
    assert len(bid) == 12 and bid == bench.conv_build_id()
    t, alg, note = bench.load_traffic(3)                       # no capture at batch 3
    assert t is None and alg is None and bid in note
    calls = []
    best, sweep = bench.pick_threads(lambda: calls.append(torch.get_num_threads()), 8)
    assert best == 8 and list(sweep) == [8] and len(calls) == 2, (best, sweep, calls)   # warm-up + one timed run per candidate


def test_bench_dump_outputs_writes_the_valid_rows(tmp_path):
    """bench.py --dump-outputs: the counts[2] valid rows of every output as float32 / float64 .npy; past the byte budget the
    same seeded subset of rows of every array, identical from run to run."""
    sys.path.insert(0, ROOT)
    import bench
    from acr_b200.ops import ParseBuffers
    B = 3
    bufs = ParseBuffers(B, "cpu")
    g = torch.Generator().manual_seed(0)
    for k in bench.PARSE_OUTPUTS:
        t = getattr(bufs, k)
        t.copy_(torch.randn(t.shape, generator=g) if t.dtype.is_floating_point else torch.randint(0, 64, t.shape, generator=g))
    bufs.counts[:3] = torch.tensor([2, 3, 5])
    mano = {"verts": torch.randn(2 * B, 778, 3, generator=g), "joints": torch.randn(2 * B, 21, 3, generator=g)}
    names = (*bench.PARSE_OUTPUTS, "verts", "joints")
    src = {k: (mano[k] if k in mano else getattr(bufs, k))[:5].numpy() for k in names}
    bench.dump_outputs(str(tmp_path / "all"), bufs, mano)
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == sorted(f"{k}.npy" for k in names + ("rows", "counts"))
    for k in names:
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype in (np.float32, np.float64) and a.shape == src[k].shape and np.array_equal(a, src[k]), k
    assert np.array_equal(np.load(tmp_path / "all" / "counts.npy"), bufs.counts.numpy())
    budget = (64 << 10) + 45000                                  # room for 4 of the 5 rows (about 10.6 KB each)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), bufs, mano, max_bytes=budget)
    rows = np.load(tmp_path / "a" / "rows.npy").astype(int)
    assert len(rows) == 4 and np.array_equal(rows, np.unique(rows)) and rows.max() < 5
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= budget
    for k in names:
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert np.array_equal(a, src[k][rows]) and np.array_equal(a, b), k


def test_lazy_outputs_refuse_stale_maps():
    from acr.model import LazyOutputs

    class FakeEngine:
        run_count = 3

        def map_nchw(self, key):
            return torch.zeros(1)
    eng = FakeEngine()
    out = LazyOutputs(eng)
    assert out["segms"].shape == (1,)
    eng.run_count += 1                                         # the arena was re-used by another forward
    assert out["segms"].shape == (1,)                          # already materialised: still there
    with pytest.raises(RuntimeError):
        out["l_center_map"]
    assert LazyOutputs(None)["segms"] is None                   # return_maps=False


def test_stem_normalisation_formula_is_bit_exact():
    """csrc/stem_tc.cu `normalised()`: x = byte as fp32, q = fma(x, rh, x * rl), out = fma(q, 2, -1) must equal the
    reference's (float)b / 255.f * 2.f - 1.f (acr/model.py:832) for every byte, bit for bit.  fp64 emulates each fma
    exactly here (24-bit x 24-bit products and their sums with one more fp32 fit in 53 bits)."""
    f32, f64 = np.float32, np.float64
    rh = np.uint32(0x3B808081).view(f32)
    rl = np.uint32(0xAF7EFEFF).view(f32)
    b = np.arange(256, dtype=np.uint32)
    x = ((b | np.uint32(0x4B000000)).view(f32) - f32(8388608.0)).astype(f32)
    assert np.array_equal(x, b.astype(f32))
    t = (x * rl).astype(f32)
    q = (x.astype(f64) * f64(rh) + t.astype(f64)).astype(f32)
    out = (q.astype(f64) * 2.0 - 1.0).astype(f32)
    ref = b.astype(f32) / f32(255.0) * f32(2.0) - f32(1.0)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    src = open(os.path.join(ROOT, "arbitrary-hands-3d-reconstruction_b200", "csrc", "stem_tc.cu")).read()
    assert "0x3B808081u" in src and "0xAF7EFEFFu" in src and "0x4B000000u" in src
