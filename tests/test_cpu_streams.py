"""Many video streams per batch, CPU side: the per-frame parse oracle and the per-stream OneEuro oracle
(tests/stream_oracle.py) against the reference (stream_golden.npz, tests/golden/make_stream_golden.py)."""
import os

import numpy as np
import pytest

from oracle import parse_ref
from tests import stream_oracle as so


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "stream_golden.npz"))


@pytest.mark.parametrize("t", range(so.T))
def test_parse_per_frame_oracle(golden, t):
    out = parse_ref_per_frame = so.parse_per_frame(so.make_stream_maps(t), so.stream_meta_ids(t))
    assert (golden["meta_ids"][t] == so.stream_meta_ids(t)).all()
    for k in ("detection_flag", "centers_pred", "reorganize_idx", "counts"):
        got, ref = np.asarray(parse_ref_per_frame[k]), golden[k][t]
        assert got.shape == ref.shape and (got == ref).all(), k
    assert (out["output_hand_type"] == np.repeat([0, 1], so.S)).all()
    for k in ("params_pred", "centers_conf"):
        assert np.abs(out[k] - golden[k][t]).max() <= 1e-6, k
    for k in ("cam", "global_orient", "hand_pose", "betas", "poses"):
        assert np.abs(out["params_dict"][k] - golden[k][t]).max() <= 5e-5, k


def test_stream_smoothing_oracle(golden):
    """One bank pair per stream, driven like acr/main.py:69-83, with a lost hand, a frame without hands and a
    reset, against the reference's filter objects (same tolerances as test_one_euro_smoothing)."""
    sm = so.StreamSmoother()
    ht = np.repeat(np.array([0, 1], np.int32), so.S)
    bi = np.concatenate([np.arange(so.S), np.arange(so.S)])
    for t in range(so.T):
        for s in so.RESETS.get(t, []):
            sm.reset(s)
        p, b = sm.apply(golden["poses"][t], golden["betas"][t], ht, golden["detection_flag"][t], bi, np.arange(so.S))
        assert np.abs(p - golden["out_poses"][t]).max() < 2e-5, t
        assert np.abs(b - golden["out_betas"][t]).max() < 1e-6, t


def test_reset_and_skipped_rows_matter(golden):
    """The fixture exercises what it was built for: without the reset, stream 2 filters differently after step 5;
    undetected rows come back unfiltered."""
    det = golden["detection_flag"]
    undet = det == 0
    assert undet.sum() == 3
    assert (golden["out_poses"][undet] == golden["poses"][undet]).all()
    sm = so.StreamSmoother()
    ht = np.repeat(np.array([0, 1], np.int32), so.S)
    bi = np.concatenate([np.arange(so.S), np.arange(so.S)])
    for t in range(so.T):
        p, _ = sm.apply(golden["poses"][t], golden["betas"][t], ht, det[t], bi, np.arange(so.S))
    rows = [2, so.S + 2]
    assert np.abs(p[rows] - golden["out_poses"][so.T - 1][rows]).max() > 1e-3


def test_batch_and_per_frame_rules_disagree():
    """On the golden's far/near step the reference's batch parse (prior decided on frame 0's far pair for the whole
    batch) and the per-frame parse (frame 1's near pair keeps its prior) really differ, on frame 1's rows only."""
    t = so.FAR_NEAR_STEP
    maps = so.make_stream_maps(t)
    batch = parse_ref.parse_maps(maps, so.stream_meta_ids(t))
    per = so.parse_per_frame(maps, so.stream_meta_ids(t))
    assert int(batch["left_hand_num"][0]) == so.S and int(batch["right_hand_num"][0]) == so.S   # same row layout here
    diff = np.abs(batch["params_pred"] - per["params_pred"]).max(1)
    assert diff[1] > 1e-3 and diff[so.S + 1] > 1e-3
    assert (diff[[0, so.S]] == 0).all()
