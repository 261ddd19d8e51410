"""ORACLE (test infrastructure, never on the product path): many video streams per batch.

numpy restatement of what the reference defines for B independent streams: each frame parsed as the
reference's ResultParser.parse parses a batch of one (oracle.parse_ref.parse at B = 1), and per stream one
pair of OneEuro filter banks applied the way acr/main.py:69-83 drives them for its single stream.  Pinned
against the reference through tests/golden/stream_golden.npz (tests/golden/make_stream_golden.py).

Row layout of a per-frame parse of B frames: row b = left hand of frame b, row B + b = its right hand.
"""
import numpy as np

from oracle import parse_ref
from oracle.rotation_ref import OneEuroBank

F = np.float32

# --------------------------------------------------------------------------- the golden's input sequence
S, T = 3, 8                 # streams, steps; slot s of every step carries stream s
SMOOTH_COEFF = 4.0
RESETS = {5: [2]}           # step -> streams that start a new clip before that step
FAR_NEAR_STEP = 2           # frame 0 a far pair, frame 1 a near pair: batch rule and per-frame rule disagree
LEFT_LOST = (3, 1)          # (step, stream): left hand not detected
NO_HAND = (4, 2)            # (step, stream): no hand at all


def stream_meta_ids(t):
    return np.arange(S, dtype=np.int64) + 100 * t


def make_stream_maps(t):
    """Seeded synthetic 64x64 maps of step t (S frames), built like the parse_golden cases: a noise centre map
    with one peak per detected hand (plus a neighbour the NMS suppresses), per-stream parameter maps that drift
    from step to step, small prior maps."""
    maps = {}
    for side in "lr":
        cm = np.empty((S, 1, 64, 64), F)
        pm = np.empty((S, 109, 64, 64), F)
        pr = np.empty((S, 106, 64, 64), F)
        for s in range(S):
            base = np.random.default_rng(1000 + 10 * s + (side == "r"))
            g = np.random.default_rng(10000 + 100 * t + 10 * s + (side == "r"))
            cm[s, 0] = g.standard_normal((64, 64)) * 0.05
            pm[s] = base.standard_normal((109, 64, 64)) + 0.3 * g.standard_normal((109, 64, 64))
            pr[s] = g.standard_normal((106, 64, 64)) * 0.1
            y, x = g.integers(0, 64, 2)
            if t == FAR_NEAR_STEP and s == 0:
                y, x = (2, 3) if side == "l" else (60, 58)
            if t == FAR_NEAR_STEP and s == 1:
                y, x = (20, 20) if side == "l" else (30, 25)
            if (t, s) == NO_HAND or ((t, s) == LEFT_LOST and side == "l"):
                continue
            cm[s, 0, y, x] = 0.9 + 0.05 * s
            if 0 < y < 63:
                cm[s, 0, y + 1, x] = 0.8
        maps[f"{side}_center_map"], maps[f"{side}_params_maps"], maps[f"{side}_prior_maps"] = cm, pm, pr
    return maps


# ------------------------------------------------------------------------------------- per-frame parse
def parse_per_frame(maps, batch_ids_meta=None):
    """parse_ref.parse at B = 1 on every frame, assembled into the fixed layout (rows b / B + b = left / right hand
    of frame b).  -> dict of (2B, ...) arrays + ``counts`` = [B, B, 2B, #true, #left, #right] + ``params_dict``."""
    B = maps["l_center_map"].shape[0]
    meta = np.arange(B) if batch_ids_meta is None else np.asarray(batch_ids_meta)
    per = [parse_ref.parse({k: v[b:b + 1] for k, v in maps.items()}, meta[b:b + 1]) for b in range(B)]
    for o in per:   # a batch of one has exactly one row per side (a detection or the dummy row)
        assert int(o["left_hand_num"][0]) == 1 and int(o["right_hand_num"][0]) == 1
    rows = lambda f: np.concatenate([np.stack([f(o)[0] for o in per]), np.stack([f(o)[1] for o in per])])
    out = dict(params_pred=rows(lambda o: o["params_pred"]), detection_flag=rows(lambda o: o["detection_flag"]),
               reorganize_idx=rows(lambda o: o["reorganize_idx"]),
               batch_ids=np.concatenate([np.arange(B), np.arange(B)]).astype(np.int64),
               centers_pred=rows(lambda o: np.concatenate([o["l_centers_pred"], o["r_centers_pred"]])),
               centers_conf=rows(lambda o: np.concatenate([o["l_centers_conf"], o["r_centers_conf"]]).reshape(-1)),
               output_hand_type=np.repeat(np.array([0, 1], np.int32), B))
    out["params_dict"] = {k: rows(lambda o: o["params_dict"][k])
                          for k in ("cam", "global_orient", "hand_pose", "betas", "poses")}
    nl, nr = int(out["detection_flag"][:B].sum()), int(out["detection_flag"][B:].sum())
    out["counts"] = np.array([B, B, 2 * B, nl + nr, nl, nr], np.int32)
    return out


# ------------------------------------------------------------------------------------ per-stream smoothing
class StreamSmoother:
    """One OneEuroBank pair (left, right) per stream, created on a stream's first detected hand or after reset()
    (the reference's create_OneEuroFilter pair of a fresh clip), applied like acr/main.py:69-83."""

    def __init__(self, smooth_coeff=SMOOTH_COEFF):
        self.c = smooth_coeff
        self.banks = {}

    def reset(self, stream):
        self.banks.pop(int(stream), None)

    def apply(self, poses, betas, hand_type, detection_flag, batch_ids, stream_ids):
        """-> smoothed copies of (n,48) poses and (n,10) betas.  Row r uses stream stream_ids[batch_ids[r]]; rows
        not detected or of a slot with a negative stream id are returned unchanged and touch no bank."""
        poses, betas = np.array(poses, F), np.array(betas, F)
        for r in range(poses.shape[0]):
            s = int(stream_ids[int(batch_ids[r])])
            if not detection_flag[r] > 0 or s < 0:
                continue
            bank = self.banks.setdefault(s, [OneEuroBank(self.c), OneEuroBank(self.c)])[int(hand_type[r] != 0)]
            poses[r], betas[r] = bank.process(poses[r], betas[r])
        return poses, betas
