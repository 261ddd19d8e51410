"""Thin Python wrappers over the C ABI for the fp32 tail of the hot path
(rotations, centre parsing, MANO).  torch only owns the memory and the stream."""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

from . import lib as L


# ----------------------------------------------------------------------------- MANO model
def pack_mano_model(asset: Dict[str, np.ndarray], flip_x: bool, device) -> torch.Tensor:
    """Pack a MANO asset (dict of numpy arrays, see acr_b200.synth.make_synthetic_mano or
    mano.assets.load_mano_pkl) into the kernel's constant layout and upload it."""
    lib = L.load()
    n = lib.acr_b200_mano_model_floats()
    out = np.zeros(n, np.float32)
    arrs = [np.ascontiguousarray(asset[k], np.float32) for k in
            ("shapedirs", "posedirs", "v_template", "J_regressor", "weights", "hands_mean")]
    assert arrs[0].shape == (778, 3, 10) and arrs[1].shape == (778, 3, 135) and arrs[2].shape == (778, 3)
    assert arrs[3].shape == (16, 778) and arrs[4].shape == (778, 16) and arrs[5].shape == (45,)
    L.check(lib.acr_b200_mano_pack_model(*[a.ctypes.data for a in arrs], int(bool(flip_x)), out.ctypes.data),
            "mano_pack_model")
    return torch.from_numpy(out).to(device)


def mano_forward(model_l: Optional[torch.Tensor], model_r: Optional[torch.Tensor], poses: torch.Tensor,
                 betas: torch.Tensor, hand_type: Optional[torch.Tensor] = None, default_side: int = 1,
                 center_idx: Optional[int] = 9, cam: Optional[torch.Tensor] = None,
                 offsets: Optional[torch.Tensor] = None, n_dev: Optional[torch.Tensor] = None,
                 want_camed: bool = True, peers=None, counts: Optional[torch.Tensor] = None):
    """-> dict(verts, joints, center[, verts_camed, pj2d, pj2d_org]); all (n, ...) fp32 CUDA tensors.
    ``peers`` (acr_b200.dist.PeerVertexGather) fuses the cross-GPU vertex all-gather into the kernel; ``counts``
    (8 int32, acr_b200_parse's row counts) then travels with the vertices."""
    dev = L.require_cuda(poses, betas, hand_type, cam, offsets, n_dev, model_l, model_r)
    n = poses.shape[0]
    poses = poses.contiguous().float()
    betas = betas.contiguous().float()
    out = dict(verts=torch.empty(n, 778, 3, device=dev), joints=torch.empty(n, 21, 3, device=dev),
               center=torch.empty(n, 1, 3, device=dev))
    if cam is not None:
        cam = cam.contiguous().float()
        if want_camed:
            out["verts_camed"] = torch.empty(n, 778, 3, device=dev)
        out["pj2d"] = torch.empty(n, 21, 2, device=dev)
        if offsets is not None:
            offsets = offsets.contiguous().float()
            out["pj2d_org"] = torch.empty(n, 21, 2, device=dev)
    if hand_type is not None:
        hand_type = hand_type.contiguous().to(torch.int32)
    if n == 0:
        return out
    lib = L.load()
    common = (L.ptr(model_l), L.ptr(model_r), L.ptr(poses), L.ptr(betas), L.ptr(hand_type),
              int(default_side), L.ptr(n_dev), n, -1 if center_idx is None else int(center_idx),
              L.ptr(cam), L.ptr(offsets), L.ptr(out["verts"]), L.ptr(out["joints"]),
              L.ptr(out["center"]), L.ptr(out.get("verts_camed")), L.ptr(out.get("pj2d")),
              L.ptr(out.get("pj2d_org")))
    with L.on(dev):
        if peers is None:
            rc = lib.acr_b200_mano_forward(*common, L.current_stream(dev))
        else:
            assert n <= peers.rows, "gather buffer too small"
            import ctypes as C
            rc = lib.acr_b200_mano_forward_gather(*common, L.ptr(counts), C.byref(peers.desc), L.current_stream(dev))
            if rc == L.OK:
                peers.note_launch()
    L.check(rc, "mano_forward")
    return out


def cam_trans(j3d: torch.Tensor, pj2d: torch.Tensor, focal_length: float = 1265.0, img_size: float = 512.0,
              n_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(n,21,3), (n,21,2) -> (n,3) camera translation (closed-form least squares on the device)."""
    dev = L.require_cuda(j3d, pj2d, n_dev)
    n = j3d.shape[0]
    out = torch.empty(n, 3, device=j3d.device)
    if n:
        with L.on(dev):
            L.check(L.load().acr_b200_cam_trans(L.ptr(j3d.contiguous().float()), L.ptr(pj2d.contiguous().float()),
                                                L.ptr(n_dev), n, float(focal_length), float(img_size), L.ptr(out),
                                                L.current_stream(dev)), "cam_trans")
    return out


class OneEuroState:
    """Device-side history of the temporal filter (one bank per hand type); zero = no history."""

    def __init__(self, device):
        self.state = torch.zeros(int(L.load().acr_b200_one_euro_state_floats()), device=device)

    def reset(self) -> None:
        self.state.zero_()


def one_euro_smooth(poses: torch.Tensor, betas: torch.Tensor, state: OneEuroState, smooth_coeff: float = 4.0,
                    hand_type: Optional[torch.Tensor] = None, detection_flag: Optional[torch.Tensor] = None,
                    n_dev: Optional[torch.Tensor] = None) -> None:
    """In-place temporal smoothing of (n,48) poses and (n,10) betas (drop-in for acr.utils.smooth_results
    applied per hand as in acr/main.py:69-83)."""
    dev = L.require_cuda(poses, betas, hand_type, detection_flag, n_dev, state.state)
    assert poses.is_contiguous() and betas.is_contiguous() and poses.dtype == betas.dtype == torch.float32
    if poses.shape[0]:
        with L.on(dev):
            L.check(L.load().acr_b200_one_euro_smooth(L.ptr(poses), L.ptr(betas), L.ptr(hand_type), L.ptr(detection_flag),
                                                      L.ptr(n_dev), poses.shape[0], L.ptr(state.state), float(smooth_coeff),
                                                      L.current_stream(dev)), "one_euro_smooth")


class StreamStates:
    """Device-side filter history of ``n_streams`` independent video streams (acr_b200_one_euro_smooth_streams):
    one OneEuroState-sized block per stream, zero = no history."""

    def __init__(self, n_streams: int, device):
        if int(n_streams) < 1:
            raise ValueError("StreamStates needs at least one stream")
        self.n_streams = int(n_streams)
        self.block = int(L.load().acr_b200_one_euro_state_floats())
        self.state = torch.zeros(self.n_streams * self.block, device=device)

    def reset(self, ids=None) -> None:
        """Forget the history of streams ``ids`` (all when None), e.g. when a stream starts a new clip.
        Enqueued on the current stream: launches already enqueued still see the old history."""
        if ids is None:
            self.state.zero_()
            return
        ids = torch.as_tensor(ids, dtype=torch.int64).reshape(-1)
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= self.n_streams):
            raise ValueError(f"stream ids must lie in [0, {self.n_streams})")
        self.state.view(self.n_streams, self.block).index_fill_(0, ids.to(self.state.device), 0.0)


def check_stream_ids(stream_ids, n_slots: Optional[int], n_streams: int) -> torch.Tensor:
    """Slot -> stream map of one batch: int32, one id per slot, a negative id (-1) for a padding slot, the others
    distinct and below ``n_streams``.  None = slot b is stream b.  Ids from the host (list, numpy, CPU tensor) are
    validated and returned as a CPU int32 tensor; a CUDA int32 tensor is returned as is, only its shape checked
    (its values stay on the device: ids outside [0, n_streams) are padding, distinct ones are the caller's duty)."""
    if stream_ids is None:
        if n_slots is None:
            raise ValueError("stream ids are required")
        stream_ids = torch.arange(n_slots, dtype=torch.int32)
    if isinstance(stream_ids, torch.Tensor) and stream_ids.is_cuda:
        if stream_ids.dtype != torch.int32 or stream_ids.dim() != 1 or \
                (n_slots is not None and stream_ids.numel() != n_slots):
            raise ValueError(f"device stream ids must be a 1-D int32 tensor with one id per slot ({n_slots})")
        return stream_ids.contiguous()
    ids = torch.as_tensor(stream_ids)
    if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
        raise TypeError(f"stream ids must be integers, got {ids.dtype}")
    if ids.dim() != 1 or (n_slots is not None and ids.numel() != n_slots):
        raise ValueError(f"stream ids: expected one id per slot ({n_slots}), got shape {tuple(ids.shape)}")
    if ids.numel() and (int(ids.min()) < -2 ** 31 or int(ids.max()) >= 2 ** 31):
        raise ValueError("stream ids must fit in int32")
    live = ids[ids >= 0]
    if live.numel() and int(live.max()) >= n_streams:
        raise ValueError(f"stream id {int(live.max())} is not below n_streams = {n_streams}")
    if live.unique().numel() != live.numel():
        raise ValueError("stream ids must be distinct within one batch (two slots of one stream would race on its "
                         "filter state)")
    return ids.to(torch.int32).cpu().contiguous()


def one_euro_smooth_streams(poses: torch.Tensor, betas: torch.Tensor, states: StreamStates, stream_ids,
                            hand_type: torch.Tensor, detection_flag: Optional[torch.Tensor], batch_ids: torch.Tensor,
                            smooth_coeff: float = 4.0, n_dev: Optional[torch.Tensor] = None) -> None:
    """In-place temporal smoothing of (n,48) poses and (n,10) betas, row r with the filter bank of stream
    ``stream_ids[batch_ids[r]]`` and hand ``hand_type[r]`` (the reference's per-frame filters of acr/main.py:69-83,
    one pair per stream).  ``stream_ids`` as in check_stream_ids: host ids are validated, a CUDA tensor is not."""
    ids = check_stream_ids(stream_ids, None, states.n_streams).to(poses.device)
    dev = L.require_cuda(poses, betas, hand_type, detection_flag, batch_ids, n_dev, ids, states.state)
    assert poses.is_contiguous() and betas.is_contiguous() and poses.dtype == betas.dtype == torch.float32
    hand_type = hand_type.contiguous().to(torch.int32)
    batch_ids = batch_ids.contiguous().to(torch.int64)
    if poses.shape[0]:
        with L.on(dev):
            L.check(L.load().acr_b200_one_euro_smooth_streams(
                L.ptr(poses), L.ptr(betas), L.ptr(hand_type), L.ptr(detection_flag), L.ptr(batch_ids), L.ptr(ids),
                states.n_streams, L.ptr(n_dev), poses.shape[0], L.ptr(states.state), float(smooth_coeff),
                L.current_stream(dev)), "one_euro_smooth_streams")


# ------------------------------------------------------------------------------ rotations
def rot6d_to_aa(rot6d: torch.Tensor) -> torch.Tensor:
    """(N, 6*J) -> (N, 3*J); drop-in for acr.utils.rot6D_to_angular."""
    dev = L.require_cuda(rot6d)
    x = rot6d.contiguous().float()
    nrot = x.numel() // 6
    out = torch.empty(x.shape[0], x.shape[1] // 2, device=x.device)
    if nrot:
        with L.on(dev):
            L.check(L.load().acr_b200_rot6d_to_aa(L.ptr(x), nrot, L.ptr(out), L.current_stream(dev)), "rot6d_to_aa")
    return out


def rodrigues(aa: torch.Tensor) -> torch.Tensor:
    """(M,3) -> (M,9); drop-in for mano.manolayer.batch_rodrigues."""
    dev = L.require_cuda(aa)
    x = aa.contiguous().float()
    out = torch.empty(x.shape[0], 9, device=x.device)
    if x.shape[0]:
        with L.on(dev):
            L.check(L.load().acr_b200_rodrigues(L.ptr(x), x.shape[0], L.ptr(out), L.current_stream(dev)), "rodrigues")
    return out


# --------------------------------------------------------------------------------- parse
class ParseBuffers:
    """Worst-case (2B rows) output buffers of acr_b200_parse, allocated once per batch size."""

    def __init__(self, B: int, device):
        f = lambda *s: torch.zeros(*s, device=device, dtype=torch.float32)
        i64 = lambda *s: torch.zeros(*s, device=device, dtype=torch.int64)
        i32 = lambda *s: torch.zeros(*s, device=device, dtype=torch.int32)
        R = 2 * B
        self.B = B
        self.params_pred, self.cam, self.global_orient = f(R, 109), f(R, 3), f(R, 3)
        self.hand_pose, self.betas, self.poses = f(R, 45), f(R, 10), f(R, 48)
        self.detection_flag, self.reorganize_idx, self.batch_ids = f(R), i64(R), i64(R)
        self.centers_pred, self.centers_conf, self.hand_type = i64(R, 2), f(R), i32(R)
        self.offsets_out, self.counts = f(R, 10), i32(8)
        self.top_idx, self.top_score, self.row_src = i32(B, 2), f(B, 2), i32(R, 4)

    def struct(self) -> L.ParseOut:
        o = L.ParseOut()
        for name, _ in L.ParseOut._fields_:
            setattr(o, name, getattr(self, name).data_ptr())
        return o


def parse_maps(maps: Dict[str, tuple], B: int, bufs: ParseBuffers, meta_batch_ids: Optional[torch.Tensor],
               offsets: Optional[torch.Tensor], conf_thresh: float = 0.35, per_frame: bool = False) -> None:
    """maps[name] = (fp32 CUDA tensor in NHWC layout, pix_stride) for l/r_center, l/r_params, l/r_prior.
    Fills ``bufs`` asynchronously on the current stream (no host sync).  ``per_frame``: every image parsed as a
    batch of one, fixed rows (b = left hand of image b, B + b = its right hand; acr_b200_parse_per_frame) instead
    of the reference's batch parse with its batch-wide rules (acr_b200_parse)."""
    lib = L.load()
    ms = []
    dev = L.require_cuda(bufs.counts, *[maps[k][0] for k in maps])
    for k in ("l_center", "r_center", "l_params", "r_params", "l_prior", "r_prior"):
        t, stride = maps[k]
        assert t.dtype == torch.float32
        m = L.Map()
        m.ptr, m.pix_stride = t.data_ptr(), int(stride)
        ms.append(m)
    if meta_batch_ids is not None:
        meta_batch_ids = meta_batch_ids.to(device=bufs.counts.device, dtype=torch.int64).contiguous()
    if offsets is not None:
        offsets = offsets.to(device=bufs.counts.device, dtype=torch.float32).contiguous()
    with L.on(dev):
        fn = lib.acr_b200_parse_per_frame if per_frame else lib.acr_b200_parse
        rc = fn(*ms, B, float(conf_thresh), L.ptr(meta_batch_ids), L.ptr(offsets), bufs.struct(), L.current_stream(dev))
    L.check(rc, "parse")
    # keep the inputs alive until the kernels have run
    bufs._keep = (meta_batch_ids, offsets, [m for m in maps.values()])
