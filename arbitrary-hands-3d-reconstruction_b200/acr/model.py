"""Drop-in ``acr.model.ACR`` (reference: /root/reference/acr/model.py:23-329, backbone :691-881).

Same constructor, ``forward(meta_data, **cfg)`` / ``head_forward(x)`` signatures, ``state_dict()``
keys (2067 tensors, checkpoint compatible) and output dict schema.  The module tree only *holds*
the parameters; the arithmetic is a precompiled CUDA launch plan (acr_b200.engine.Engine).
"""
from __future__ import annotations

import logging
from collections import OrderedDict

import torch
import torch.nn as nn

from acr.config import args
from acr.result_parser import ResultParser
from acr_b200.engine import Engine
from acr_b200.netspec import WIDTHS, WIDTHS_W48, build_acr_spec

BN_MOMENTUM = 0.1
_MAP_KEYS = ('l_params_maps', 'r_params_maps', 'l_center_map', 'r_center_map', 'l_prior_maps', 'r_prior_maps', 'segms')


class _Node(nn.Module):
    """Anonymous container so that parameters get the reference's dotted names."""


def _attach(root: nn.Module, dotted: str, tensor: torch.Tensor, is_param: bool) -> None:
    parts = dotted.split('.')
    m = root
    for p in parts[:-1]:
        if not hasattr(m, p) or getattr(m, p) is None:
            m.add_module(p, _Node())
        m = getattr(m, p)
    if is_param:
        m.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))
    else:
        m.register_buffer(parts[-1], tensor)


class LazyOutputs(dict):
    """``outputs`` dict whose seven map entries are converted from the engine's NHWC arena to the
    reference's fp32 NCHW tensors on first access (nothing on the hot path reads them; at batch 256 the
    seven maps are 2.9 GB in the reference's layout).  The arena is re-used by the next forward of the
    same batch size, so a map that was NOT read before that next forward is gone: reading it then raises
    instead of silently returning the newer frame's data.  ``materialize()`` converts all seven now."""

    def __init__(self, engine, *a, **k):
        super().__init__(*a, **k)
        self._engine = engine
        self._run = engine.run_count if engine is not None else 0
        for key in _MAP_KEYS:
            dict.__setitem__(self, key, None)

    def __getitem__(self, key):
        v = dict.__getitem__(self, key)
        if v is None and key in _MAP_KEYS and self._engine is not None:
            if self._engine.run_count != self._run:
                raise RuntimeError(f"outputs['{key}'] was not read before the next forward of this batch size "
                                   "re-used the activation arena; call outputs.materialize() right after forward() "
                                   "to keep the maps across frames")
            v = self._engine.map_nchw(key)
            dict.__setitem__(self, key, v)
        return v

    def materialize(self):
        for key in _MAP_KEYS:
            self[key]
        return self

    def get(self, key, default=None):
        return self[key] if key in self else default

    def items(self):
        return [(k, self[k]) for k in self.keys()]

    def values(self):
        return [self[k] for k in self.keys()]


class ACR(nn.Module):
    def __init__(self, **kwargs):
        super().__init__()
        self._widths = {32: WIDTHS, 48: WIDTHS_W48}[int(getattr(args(), 'hrnet_width', 32))]
        self._spec = build_acr_spec(args().input_size, widths=self._widths)
        g = torch.Generator().manual_seed(0)
        for key, (shape, kind) in self._spec.params.items():
            if kind == 'bn_nbt':
                t = torch.zeros(shape, dtype=torch.long)
            elif kind == 'bn_var' or kind == 'bn_w':
                t = torch.ones(shape)
            elif kind in ('bn_mean', 'bn_b', 'conv_b', 'lin_b'):
                t = torch.zeros(shape)
            else:
                t = torch.randn(shape, generator=g) * 0.01
            _attach(self, key, t, is_param=kind not in ('bn_mean', 'bn_var', 'bn_nbt'))
        self._result_parser = ResultParser()
        self.outmap_size = args().centermap_size
        self._engines = OrderedDict()     # LRU of launch plans, keyed by (batch, device, dtype, flags, heads-only)
        self._blobs = {}                  # packed weights, shared by every plan of one (device, dtype, flags)
        self.max_engines = int(kwargs.get('max_engines', 3))
        self.debug_ref_conv = bool(kwargs.get('debug_ref_conv', False))

    # ------------------------------------------------------------------ engine
    def invalidate_engine(self):
        self._engines = OrderedDict()
        self._blobs = {}

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self.invalidate_engine()
        return r

    _warned_fp32 = False

    def _act_dtype(self):
        """'bf16' / 'fp16': 16-bit storage, fp32 accumulation on the tensor cores (fp16 is the reference's
        autocast mode, acr/model.py:36-41).  'fp32' (the reference's shipped default, configs/demo.yml:7):
        the validation plan -- fp32 storage, fp64 accumulation on the CUDA cores -- reference-accurate
        (1e-4 end to end) but ~100x slower than the 16-bit plans."""
        p = args().model_precision
        if p == 'bf16':
            return torch.bfloat16
        if p == 'fp16':
            return torch.float16
        if p == 'fp32':
            if not ACR._warned_fp32:
                logging.warning("model_precision='fp32' runs the fp32 validation plan on the CUDA cores (reference-"
                                "accurate, slow); use 'fp16' (the reference's autocast mode) or 'bf16' for throughput")
                ACR._warned_fp32 = True
            return torch.float32
        raise ValueError(f"model_precision must be 'fp32', 'fp16' or 'bf16', got {p!r}")

    def engine(self, batch: int, device, head_only: bool = False) -> Engine:
        """Launch plan for this batch size (built on first use).  Plans share one packed weight blob per
        (device, dtype); at most ``max_engines`` plans (each owns a ~26 MiB/image activation arena) are kept,
        least recently used first out -- variable batch sizes (the last partial batch of a video) do not
        accumulate GPU memory."""
        dt = self._act_dtype()
        dev = torch.device(device)
        if dev.type == 'cuda' and dev.index is None:
            dev = torch.device('cuda', torch.cuda.current_device())
        bkey = (str(dev), dt, self.debug_ref_conv, head_only)
        key = (batch,) + bkey
        if key in self._engines:
            self._engines.move_to_end(key)
            return self._engines[key]
        eng = Engine(self.state_dict(), batch, dev, dt, args().input_size, debug_ref_conv=self.debug_ref_conv,
                     head_only=head_only, weights=self._blobs.get(bkey), widths=self._widths)
        self._blobs[bkey] = eng.weights
        self._engines[key] = eng
        while len(self._engines) > max(1, self.max_engines):
            self._engines.popitem(last=False)
        return eng

    # ----------------------------------------------------------------- forward
    def _image(self, meta_data):
        dev = next(self.parameters()).device
        if dev.type != 'cuda':
            raise RuntimeError("acr.model.ACR runs on a CUDA device only: call .cuda() first (no CPU fallback)")
        img = meta_data['image']
        if img.dtype != torch.uint8:      # the reference accepts float 0..255 too
            img = img.round().clamp(0, 255).to(torch.uint8)
        return img.to(dev, non_blocking=True).contiguous(), dev

    @torch.no_grad()
    def forward(self, meta_data, **cfg):
        img, dev = self._image(meta_data)
        eng = self.engine(img.shape[0], dev)
        eng.run(img)
        outputs = LazyOutputs(eng if args().return_maps else None)
        bufs = self._result_parser.launch(eng.parse_inputs(), img.shape[0], meta_data, dev)
        outputs, meta_data = self._result_parser.collect(bufs, outputs, meta_data)
        outputs['meta_data'] = meta_data
        return outputs

    @torch.no_grad()
    def forward_dense(self, meta_data, per_frame=False):
        """Sync-free variant for the fused pipeline: runs backbone + heads + parse and returns the
        engine and the worst-case (2B rows) parse buffers; row validity lives in ``bufs.counts``.
        ``per_frame``: every image parsed as a batch of one, rows b / B + b = left / right hand of image b.
        ZERO COPY: the returned buffers are the per-batch-size cached ones and alias the next call's
        results -- consume (or copy) them before the next forward of the same batch size."""
        img, dev = self._image(meta_data)
        eng = self.engine(img.shape[0], dev)
        eng.run(img)
        bufs = self._result_parser.launch(eng.parse_inputs(), img.shape[0], meta_data, dev, per_frame=per_frame)
        return eng, bufs

    @torch.no_grad()
    def head_forward(self, x, gt_segm=None):
        """Reference: /root/reference/acr/model.py:47-65.  x (B,32,128,128) backbone feature -> dict of the seven
        maps, all fp32 NCHW: SegmNet, coord concat, global heads, part branch.  Runs the heads-only launch
        plan (the ops after the trunk); ``gt_segm`` is accepted and ignored like in the reference."""
        dev = next(self.parameters()).device
        if dev.type != 'cuda':
            raise RuntimeError("acr.model.ACR runs on a CUDA device only: call .cuda() first (no CPU fallback)")
        eng = self.engine(x.shape[0], dev, head_only=True)
        eng.run_heads(x.to(dev))
        return {k: eng.map_nchw(k) for k in ('l_params_maps', 'r_params_maps', 'l_center_map', 'r_center_map',
                                             'l_prior_maps', 'r_prior_maps', 'segms')}
