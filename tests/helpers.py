"""Shared helpers for the parity tests (single-op harness around the C ABI)."""
import ctypes as C
import os

import numpy as np
import torch

from acr_b200 import lib as L

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rup(x, m):
    return (x + m - 1) // m * m


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-12))


def to_nhwc_padded(x_nchw: torch.Tensor, stride: int, dtype) -> torch.Tensor:
    """(B,C,H,W) float -> (B,H,W,stride) `dtype`, zero padded channels."""
    B, Cc, H, W = x_nchw.shape
    out = torch.zeros(B, H, W, stride, dtype=dtype)
    out[..., :Cc] = x_nchw.permute(0, 2, 3, 1).to(dtype)
    return out


def ctensor(offset, Cc, H, W, stride, dt, external=0):
    t = L.Tensor()
    t.offset, t.C, t.H, t.W, t.pix_stride, t.dtype, t.external = offset, Cc, H, W, stride, dt, external
    return t


def pack_conv_host(w, conv_bias, bn, cin_pad, cout_pad, dt):
    """-> (packed uint16 (cout_pad,k*k,cin_pad), bias fp32 (cout_pad)) via the library's host packer."""
    lib = L.load()
    w = np.ascontiguousarray(w, np.float32)
    cout, cin, k, _ = w.shape
    wp = np.zeros((cout_pad, k * k, cin_pad), np.uint16)
    bias = np.zeros(cout_pad, np.float32)
    p = lambda a: None if a is None else np.ascontiguousarray(a, np.float32).ctypes.data
    keep = [None if a is None else np.ascontiguousarray(a, np.float32) for a in ([conv_bias] + list(bn or [None] * 4))]
    q = lambda a: None if a is None else a.ctypes.data
    L.check(lib.acr_b200_pack_conv(w.ctypes.data, q(keep[0]), q(keep[1]), q(keep[2]), q(keep[3]), q(keep[4]),
                                   1e-5, cout, cin, k, cout_pad, cin_pad, dt, wp.ctypes.data, bias.ctypes.data),
            "pack_conv")
    return wp, bias


def u16_to_float(a: np.ndarray, dt) -> torch.Tensor:
    t = torch.from_numpy(a.view(np.int16).copy())
    return t.view(torch.bfloat16 if dt == L.DT_BF16 else torch.float16).float()


def run_conv_case(kind, B, H, W, cin, cout, k, s, relu, residual, bias, bn, out_f32, dt=L.DT_BF16, seed=0,
                  in_stride=None, cin_pad=None):
    """Runs one conv through acr_b200_run_op on the GPU and returns (got, expected) fp32 NCHW."""
    import torch.nn.functional as Fn
    g = torch.Generator().manual_seed(seed)
    tdt = torch.bfloat16 if dt == L.DT_BF16 else torch.float16
    in_stride = in_stride or rup(cin, 16)
    cin_pad, cout_pad = cin_pad or rup(cin, 16), rup(cout, 16)
    Ho, Wo = H // s, W // s
    x = torch.randn(B, cin, H, W, generator=g)
    w = torch.randn(cout, cin, k, k, generator=g) * (2.0 / (cin * k * k)) ** 0.5
    cb = torch.randn(cout, generator=g) * 0.1 if bias else None
    bnp = None
    if bn:
        bnp = [torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g) * 0.1,
               torch.randn(cout, generator=g) * 0.1, torch.rand(cout, generator=g) + 0.5]
    wp, bvec = pack_conv_host(w.numpy(), None if cb is None else cb.numpy(),
                              None if bnp is None else [t.numpy() for t in bnp], cin_pad, cout_pad, dt)
    xin = to_nhwc_padded(x, in_stride, tdt)
    res = torch.randn(B, cout, Ho, Wo, generator=g) if residual else None
    # arena layout: [x | res | out]
    esz = 2
    off_x = 0
    off_r = rup(xin.numel() * esz, 1024)
    res_stride = cout_pad
    rbytes = B * Ho * Wo * res_stride * esz if residual else 0
    off_o = rup(off_r + rbytes, 1024)
    oesz = 4 if out_f32 else 2
    obytes = B * Ho * Wo * cout_pad * oesz
    arena = torch.zeros(off_o + obytes + 1024, dtype=torch.uint8)
    arena[off_o: off_o + obytes] = 0xFF      # NaN: a channel the kernel does not write (pad channels included) stays NaN
    arena[off_x: off_x + xin.numel() * esz] = xin.view(torch.uint8).flatten()
    if residual:
        rin = to_nhwc_padded(res, res_stride, tdt)
        arena[off_r: off_r + rin.numel() * esz] = rin.view(torch.uint8).flatten()
    blob = np.concatenate([wp.view(np.uint8).reshape(-1), np.zeros((-wp.nbytes) % 256, np.uint8),
                           bvec.view(np.uint8).reshape(-1)])
    w_off, b_off = 0, wp.nbytes + ((-wp.nbytes) % 256)
    op = L.Op()
    op.kind = kind
    op.n_in = 2 if residual else 1
    op.in_[0] = ctensor(off_x, cin, H, W, in_stride, dt)
    if residual:
        op.in_[1] = ctensor(off_r, cout, Ho, Wo, res_stride, dt)
    op.out = ctensor(off_o, cout, Ho, Wo, cout_pad, L.DT_F32 if out_f32 else dt)
    op.w_offset[0], op.w_offset[1] = w_off, b_off
    op.k, op.stride, op.relu, op.has_residual = k, s, int(relu), int(residual)
    op.cin_pad, op.cout_pad = cin_pad, cout_pad
    d_arena = arena.cuda()
    d_blob = torch.from_numpy(blob).cuda()
    lib = L.load()
    L.check(lib.acr_b200_run_op(C.byref(op), B, d_arena.data_ptr(), d_blob.data_ptr(), None, dt,
                                torch.cuda.current_stream().cuda_stream), "run_op")
    torch.cuda.synchronize()
    raw = d_arena[off_o: off_o + obytes].cpu()
    got = raw.view(torch.float32 if out_f32 else tdt).view(B, Ho, Wo, cout_pad).float()
    pad_ok = bool((got[..., cout:] == 0).all())
    got = got[..., :cout].permute(0, 3, 1, 2).contiguous()
    # expected: same rounded operands, fp32 math on the CPU
    wf = u16_to_float(wp, dt).view(cout_pad, k, k, cin_pad)[:cout, :, :, :cin].permute(0, 3, 1, 2).contiguous()
    xf = xin[..., :cin].float().permute(0, 3, 1, 2).contiguous()
    exp = Fn.conv2d(xf, wf, torch.from_numpy(bvec[:cout].copy()), s, k // 2)
    if residual:
        exp = exp + rin[..., :cout].float().permute(0, 3, 1, 2)
    if relu:
        exp = torch.relu(exp)
    return got, exp, pad_ok
