"""Drop-in ``ResultParser`` (reference: /root/reference/acr/result_parser.py:7-190).

``parse(outputs, meta_data, cfg)`` takes the reference's dict of NCHW maps; inside the fused
pipeline ``parse_engine`` reads the engine's NHWC fp32 maps in place.  Either way the work is three
small kernels (acr_b200_parse) and exactly one device->host read (the two hand counts) instead
of the reference's >=6 implicit syncs.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from acr.config import args
from acr_b200 import ops as _ops


class ResultParser(nn.Module):
    def __init__(self):
        super().__init__()
        self.map_size = args().centermap_size
        self.part_name = ['cam', 'global_orient', 'hand_pose', 'betas']
        self.part_idx = [args().cam_dim, args().rot_dim, (args().mano_theta_num - 1) * args().rot_dim, 10]
        self.kps_num = 21
        self.params_num = int(np.array(self.part_idx).sum())
        if (args().prior_mode, args().inter_prior, args().Rot_type, self.map_size) != ('cross', True, '6D', 64):
            raise ValueError("only prior_mode='cross', inter_prior=True, Rot_type='6D', centermap_size=64 "
                             "(the reference's shipped configuration) are supported")
        self._pbufs = {}

    def _parse_buffers(self, B, device, per_frame=False):
        key = (B, str(device), per_frame)
        if key not in self._pbufs:
            self._pbufs[key] = _ops.ParseBuffers(B, device)
        return self._pbufs[key]

    # ------------------------------------------------------------------ kernels
    def launch(self, maps, B, meta_data, device, per_frame=False):
        """Enqueue the parse kernels; returns the worst-case buffers (no sync).  ``per_frame``: each image parsed
        as a batch of one into fixed rows (independent video streams), see acr_b200.ops.parse_maps."""
        bufs = self._parse_buffers(B, device, per_frame)
        ids = meta_data.get('batch_ids') if meta_data is not None else None
        offs = meta_data.get('offsets') if meta_data is not None else None
        _ops.parse_maps(maps, B, bufs, ids, offs, args().centermap_conf_thresh, per_frame=per_frame)
        return bufs

    @staticmethod
    def collect(bufs, outputs, meta_data):
        """One D2H read of (L, R), then copy the N valid rows of the (per batch size cached, worst-case sized)
        parse buffers into fresh tensors with the reference's output schema.  Like the reference, every call
        returns its own tensors: a later forward() does not overwrite them and the in-place temporal smoothing
        of acr.main works on this call's rows only.  (The sync-free ``forward_dense`` / ``fused_forward`` path
        hands out the shared buffers themselves -- zero copy -- and documents that.)"""
        L, R = (int(v) for v in bufs.counts[:2].tolist())
        N = L + R
        own = lambda t: t[:N].clone()
        params_pred = own(bufs.params_pred)
        outputs['params_pred'] = params_pred
        outputs['l_params_pred'], outputs['r_params_pred'] = params_pred[:L], params_pred[L:N]
        outputs['detection_flag'] = own(bufs.detection_flag)
        outputs['detection_flag_cache'] = outputs['detection_flag'].bool()
        centers, conf = own(bufs.centers_pred), own(bufs.centers_conf)
        outputs['l_centers_pred'], outputs['r_centers_pred'] = centers[:L], centers[L:N]
        outputs['l_centers_conf'] = conf[:L].unsqueeze(1)
        outputs['r_centers_conf'] = conf[L:N].unsqueeze(1)
        dev = bufs.counts.device
        outputs['left_hand_num'] = torch.tensor([L], device=dev)
        outputs['right_hand_num'] = torch.tensor([R], device=dev)
        outputs['reorganize_idx'] = own(bufs.reorganize_idx)
        outputs['output_hand_type'] = own(bufs.hand_type)
        outputs['params_dict'] = dict(cam=own(bufs.cam), global_orient=own(bufs.global_orient),
                                      hand_pose=own(bufs.hand_pose), betas=own(bufs.betas), poses=own(bufs.poses))
        if meta_data is not None:
            bi = own(bufs.batch_ids)
            for key in ('image', 'offsets', 'imgpath'):      # result_parser.py:186-187
                if key in meta_data:
                    v = meta_data[key]
                    if isinstance(v, torch.Tensor):
                        meta_data[key] = v[bi.to(v.device)]
                    elif isinstance(v, list):
                        meta_data[key] = np.array(v)[bi.cpu().numpy()]
        return outputs, meta_data

    # ---------------------------------------------------------- reference entry
    @torch.no_grad()
    def parse(self, outputs, meta_data, cfg=None):
        """Reference signature: NCHW fp32 maps in ``outputs`` (result_parser.py:21-40)."""
        names = dict(l_center='l_center_map', r_center='r_center_map', l_params='l_params_maps',
                     r_params='r_params_maps', l_prior='l_prior_maps', r_prior='r_prior_maps')
        maps = {}
        for k, n in names.items():
            t = outputs[n].float().permute(0, 2, 3, 1).contiguous()
            maps[k] = (t, t.shape[-1])
        B = outputs['l_center_map'].shape[0]
        bufs = self.launch(maps, B, meta_data, outputs['l_center_map'].device)
        return self.collect(bufs, outputs, meta_data)
