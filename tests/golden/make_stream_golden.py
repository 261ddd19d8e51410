#!/usr/bin/env python
"""Generate tests/golden/stream_golden.npz by running the UNMODIFIED reference (make_golden.import_reference) on the seeded
synthetic sequence of tests/stream_oracle.py: S = 3 streams x T = 8 steps of 64x64 maps.  Each frame goes
through ResultParser.parse as a batch of one (the reference's video mode, acr/main.py:183-201), then its two
rows through smooth_results with the stream's own create_OneEuroFilter pair, as process_results
(acr/main.py:69-83) drives the filters of its single stream (on copies of the rows, see below).  A reset is a
fresh create_OneEuroFilter pair.

    python tests/golden/make_stream_golden.py

Rows are stored in the per-frame layout: row s = left hand of frame s, row S + s = its right hand.  The maps are
not stored (21 MB a step); tests rebuild them with tests/stream_oracle.make_stream_maps.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import import_reference  # noqa: E402


def main():
    torch = import_reference()
    from tests import stream_oracle as so
    import acr.utils as ref_utils
    from acr.result_parser import ResultParser
    rp = ResultParser()
    S, T = so.S, so.T
    g = {k: [] for k in ("params_pred", "detection_flag", "reorganize_idx", "centers_pred", "centers_conf", "counts",
                         "cam", "global_orient", "hand_pose", "betas", "poses", "out_poses", "out_betas")}
    filters = {}
    for t in range(T):
        for s in so.RESETS.get(t, []):
            filters.pop(s, None)
        maps = so.make_stream_maps(t)
        meta_ids = so.stream_meta_ids(t)
        per = []
        for s in range(S):
            outs = {k: torch.from_numpy(v[s:s + 1].copy()) for k, v in maps.items()}
            meta = {"batch_ids": torch.tensor([meta_ids[s]]), "offsets": torch.zeros(1, 10), "image": torch.zeros(1, 1)}
            o, _ = rp.parse(outs, meta, {})
            assert int(o["left_hand_num"]) == 1 and int(o["right_hand_num"]) == 1
            pd = o["params_dict"]
            raw = (pd["poses"].clone(), pd["betas"].clone())
            # acr/main.py:69-83 on this stream's filters (row index = hand type at a batch of one).  The rows are
            # handed over as copies, like smooth_golden.npz does: process_results passes views of the rows it then
            # overwrites, and LowPassFilter keeps a reference to its input, so from a clip's third frame on the
            # reference's pose / betas derivative would be taken against the previous FILTERED value.  The device
            # filter (acr_b200_one_euro_smooth, pinned by smooth_golden.npz) keeps the raw value, as the filter means.
            f = filters.setdefault(s, {0: ref_utils.create_OneEuroFilter(so.SMOOTH_COEFF),
                                       1: ref_utils.create_OneEuroFilter(so.SMOOTH_COEFF)})
            for sid, flag in enumerate(o["detection_flag_cache"]):
                if flag:
                    pd["poses"][sid], pd["betas"][sid] = ref_utils.smooth_results(f[sid], pd["poses"][sid].clone(),
                                                                                  pd["betas"][sid].clone())
            per.append(dict(params_pred=o["params_pred"].numpy(), detection_flag=o["detection_flag"].float().numpy(),
                            reorganize_idx=o["reorganize_idx"].numpy(),
                            centers_pred=torch.cat([o["l_centers_pred"], o["r_centers_pred"]]).numpy(),
                            centers_conf=torch.cat([o["l_centers_conf"], o["r_centers_conf"]]).reshape(-1).numpy(),
                            cam=pd["cam"].numpy(), global_orient=pd["global_orient"].numpy(),
                            hand_pose=pd["hand_pose"].numpy(), poses=raw[0].numpy(), betas=raw[1].numpy(),
                            out_poses=pd["poses"].numpy(), out_betas=pd["betas"].numpy()))
        for k in g:
            if k == "counts":
                continue
            g[k].append(np.concatenate([np.stack([p[k][0] for p in per]), np.stack([p[k][1] for p in per])]))
        nl = int(sum(p["detection_flag"][0] for p in per))
        nr = int(sum(p["detection_flag"][1] for p in per))
        g["counts"].append(np.array([S, S, 2 * S, nl + nr, nl, nr], np.int32))
    out = {k: np.stack(v) for k, v in g.items()}
    out["meta_ids"] = np.stack([so.stream_meta_ids(t) for t in range(T)])
    out["resets"] = np.array([(t, s) for t, ss in so.RESETS.items() for s in ss], np.int64)
    # the sequence must hold the cases it was designed for
    det = out["detection_flag"]
    assert det[so.LEFT_LOST[0], so.LEFT_LOST[1]] == 0 and det[so.LEFT_LOST[0], S + so.LEFT_LOST[1]] == 1
    assert det[so.NO_HAND[0], so.NO_HAND[1]] == 0 and det[so.NO_HAND[0], S + so.NO_HAND[1]] == 0
    assert det.sum() == 2 * S * T - 3, det
    np.savez_compressed(os.path.join(HERE, "stream_golden.npz"), **out)
    print("stream_golden:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
