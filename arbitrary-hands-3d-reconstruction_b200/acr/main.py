"""Drop-in application wrapper ``acr.main.ACR`` (reference: /root/reference/acr/main.py:24-141),
hot path only: model -> parse -> MANO.  Rendering / visualisation / CLI loops are out of scope."""
from __future__ import annotations

import torch
import torch.nn as nn

from acr.config import args
from acr.mano_wrapper import MANOWrapper
from acr.model import ACR as ACR_v1
from acr.utils import justify_detection_state, load_model


class ACR(nn.Module):
    def __init__(self, args_set=None, state_dict=None, mano_assets=None):
        super().__init__()
        self.demo_cfg = {'mode': 'parsing', 'calc_loss': False}
        cfg = vars(args() if args_set is None else args_set)
        for k, v in cfg.items():
            setattr(self, k, v)
        self._build_model_(state_dict, mano_assets)

    def _build_model_(self, state_dict, mano_assets):
        model = ACR_v1().eval()
        if state_dict is not None:
            model.load_state_dict(state_dict, strict=True)
        else:
            model = load_model(self.model_path, model, prefix='module.', drop_prefix='', fix_loaded=False)
        self.model = model.cuda()
        self.mano_regression = MANOWrapper(mano_assets).cuda()

    @torch.no_grad()
    def process_results(self, outputs):
        # temporal optimisation (acr/main.py:69-83): OneEuro filters on poses / betas, one bank per hand type,
        # applied between parse and MANO -- here one device kernel instead of host-side filter objects
        if getattr(self, 'temporal_optimization', False):
            from acr_b200 import ops as _ops
            pd = outputs['params_dict']
            assert len(pd['poses']) == 2, 'temporal smoothing streams one frame (two hand slots) at a time'
            if getattr(self, '_one_euro', None) is None:
                self._one_euro = _ops.OneEuroState(pd['poses'].device)
            poses, betas = pd['poses'].contiguous(), pd['betas'].contiguous()
            _ops.one_euro_smooth(poses, betas, self._one_euro, float(self.smooth_coeff),
                                 hand_type=outputs['output_hand_type'], detection_flag=outputs['detection_flag_cache'].float())
            pd['poses'], pd['betas'] = poses, betas
        outputs = self.mano_regression(outputs, outputs['meta_data'])
        return outputs

    @torch.no_grad()
    def batch_forward(self, images_rgb_u8, offsets=None, batch_ids=None):
        """B frames (uint8 BHWC RGB, already 512x512) -> reference-schema outputs incl. MANO."""
        B = images_rgb_u8.shape[0]
        if offsets is None:
            offsets = torch.tensor([[512., 512, 0, 0, 0, 0, 0, 0, 0, 0]]).repeat(B, 1)
        meta = {'image': images_rgb_u8, 'offsets': offsets,
                'batch_ids': torch.arange(B) if batch_ids is None else batch_ids}
        outputs = self.model(meta, **self.demo_cfg)
        return self.process_results(outputs)

    @torch.no_grad()
    def fused_forward(self, images_rgb_u8, offsets, out=None, peers=None):
        """Sync-free pipeline: backbone + heads + parse + MANO enqueued back to back; MANO runs over
        the worst case 2B rows and skips rows >= L+R on the device.  Returns dense buffers (zero copy: the
        parse buffers are shared per batch size, consume them before the next call).  ``peers``
        (acr_b200.dist.PeerVertexGather): the MANO kernel also stores vertices and row counts into every
        rank's gather buffer."""
        meta = {'image': images_rgb_u8, 'offsets': offsets, 'batch_ids': None}
        eng, bufs = self.model.forward_dense(meta)
        return bufs, self._mano_dense(bufs, peers)

    def _mano_dense(self, bufs, peers=None):
        """MANO (+ cam_trans) over the 2B rows of dense parse buffers; rows >= counts[2] are skipped on the device."""
        from acr_b200 import ops as _ops
        ml, mr = self.mano_regression.models()
        mano = _ops.mano_forward(ml, mr, bufs.poses, bufs.betas, bufs.hand_type, 1, self.mano_regression.center_idx,
                                 bufs.cam, bufs.offsets_out, n_dev=bufs.counts[2:3], peers=peers, counts=bufs.counts)
        if args().cam_trans_mode == 'lstsq':
            mano['cam_trans'] = _ops.cam_trans(mano['joints'], mano['pj2d'], args().focal_length, 512.0,
                                               n_dev=bufs.counts[2:3])
        return mano

    @torch.no_grad()
    def stream_forward(self, images_rgb_u8, offsets, streams=None, stream_ids=None):
        """B frames of B independent video streams in one sync-free pass: backbone + heads, per-frame parse (every
        frame parsed as the reference parses it alone; row b = left hand of frame b, row B + b = its right hand,
        all 2B rows valid), then -- when ``streams`` (acr_b200.ops.StreamStates) is given -- OneEuro smoothing with
        ``smooth_coeff``, each frame with its own stream's filters, then MANO over the 2B rows and cam_trans.
        ``stream_ids``: stream of each slot (int32, length B; -1 = padding slot, not smoothed); None = slot b is
        stream b.  Host ids are validated (distinct, below n_streams); a CUDA int32 tensor is used as is.  Returns
        ``(bufs, mano)`` with fused_forward's zero-copy contract."""
        from acr_b200 import ops as _ops
        B = images_rgb_u8.shape[0]
        if streams is not None:      # validate before any launch
            ids = _ops.check_stream_ids(stream_ids, B, streams.n_streams)
        meta = {'image': images_rgb_u8, 'offsets': offsets, 'batch_ids': None}
        eng, bufs = self.model.forward_dense(meta, per_frame=True)
        if streams is not None:
            _ops.one_euro_smooth_streams(bufs.poses, bufs.betas, streams, ids.to(bufs.poses.device),
                                         hand_type=bufs.hand_type, detection_flag=bufs.detection_flag,
                                         batch_ids=bufs.batch_ids, smooth_coeff=float(self.smooth_coeff))
        return bufs, self._mano_dense(bufs)

    @torch.no_grad()
    def capture_graph(self, batch: int, device=None, streams=None):
        """CUDA-graph the whole sync-free pipeline (backbone + heads + parse + MANO + cam_trans, ~380 kernel
        launches) for a fixed batch size: returns ``replay(frames_u8, offsets) -> (bufs, mano)`` that copies
        the inputs into static buffers and launches ONE graph.  This is what makes the reference's
        frame-by-frame video / webcam loop (acr/main.py:183-201, batch 1) latency-bound by the GPU instead
        of by ~380 host-side launches.  ``streams`` (acr_b200.ops.StreamStates): the graph is stream_forward
        instead (per-frame parse + per-stream smoothing, state on the device), and
        ``replay(frames_u8, offsets, stream_ids=None)`` also copies the slot -> stream ids (None: slot b is stream
        b) into a static buffer."""
        from acr_b200 import ops as _ops
        dev = torch.device(device) if device is not None else next(self.model.parameters()).device
        frames = torch.zeros(batch, args().input_size, args().input_size, 3, dtype=torch.uint8, device=dev)
        offsets = torch.zeros(batch, 10, device=dev)
        if streams is None:
            run = lambda: self.fused_forward(frames, offsets)
        else:
            ids = torch.full((batch,), -1, dtype=torch.int32, device=dev)     # warm-up: padding only, no state touched
            run = lambda: self.stream_forward(frames, offsets, streams, ids)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                       # warm-up: builds the engine, sets func attributes
            for _ in range(2):
                run()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            bufs, mano = run()

        def replay(frames_u8, offs, stream_ids=None):
            frames.copy_(frames_u8, non_blocking=True)
            offsets.copy_(offs, non_blocking=True)
            if streams is not None:
                ids.copy_(_ops.check_stream_ids(stream_ids, batch, streams.n_streams))
            elif stream_ids is not None:
                raise ValueError("stream_ids needs a graph captured with streams=")
            graph.replay()
            return bufs, mano

        replay.graph, replay.static_inputs = graph, (frames, offsets) if streams is None else (frames, offsets, ids)
        return replay

    @torch.no_grad()
    def single_image_forward(self, image_rgb_u8_512, path=None):
        meta = {'image': image_rgb_u8_512[None] if image_rgb_u8_512.dim() == 3 else image_rgb_u8_512,
                'offsets': torch.tensor([[512., 512, 0, 0, 0, 0, 0, 0, 0, 0]]), 'batch_ids': torch.arange(1)}
        outputs = self.model(meta, **self.demo_cfg)
        outputs['detection_flag'], outputs['reorganize_idx'] = justify_detection_state(
            outputs['detection_flag'], outputs['reorganize_idx'])
        outputs['meta_data']['imgpath'] = [path]
        return outputs
