"""GPU: the persistent tile loop of the tcgen05 conv (csrc/conv_tc.cu) against a float64 reference, at every kernel
instance the product plans launch.

A CTA of conv_tc_kernel walks the virtual tiles blockIdx.x, blockIdx.x + gridDim.x, ... (super-tile x N split).  The TMEM
buffer alternation, the A/B stage and TMEM barrier phases, the staged epilogue's residual prefetch and slab ring and the
per-tile N offset of split layers only run from a CTA's second tile on, and the grid is one CTA per SM, so the small
op-level cases of test_gpu_conv.py never get there.  Here every case runs on B >= 3 images of distinct content at several
grid caps (ACR_B200_CONV_MAX_CTAS): unset, 3, 4 and 5 CTAs -- >= 3 tiles per CTA, odd grids, grids that do not divide
the tile count, and for N-split layers CTAs that alternate between the two halves.

Reference: float64 convolution of the identically rounded operands (the 16-bit weights unpacked from the packed blob).
Bound, per element, derived from the fp32 arithmetic of the kernel rather than tuned: with K products accumulated,
A = conv(|x|, |w|) + |bias| and one rounding (2^-24) per addition, the pre-activation error is <= (K + 1) 2^-24 A; the
residual and every extra term add one rounding each (of |res| + sum |ext| + the running magnitude); 1.1**x propagates
its input error through exp and adds powf's 4 ulp; a 16-bit output adds the final rounding u |ref| (u = 2^-8 bf16, 2^-11
fp16; plus half the fp16 subnormal spacing).

Sentinels: the whole arena starts as random bytes, the output region as NaN; afterwards every logical output channel must be
finite and within its bound, every pad channel exactly +0 (it is the K padding of the next conv: stale NaN x 0 = NaN),
and every byte outside the output (inputs, residual, extra terms, guards) unchanged.  Summation order inside a tile does not
depend on the CTA that runs it, so the output must be bit-identical at every grid cap."""
import ctypes as C
import math
import os
import zlib
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from acr_b200 import lib as L
from tests.helpers import ctensor, rup

pytestmark = pytest.mark.gpu

CAP_ENV = "ACR_B200_CONV_MAX_CTAS"
CAPS = (None, 3, 4, 5)        # None = one CTA per SM (the product grid)
DEPTH_CAP = 3                 # the cap at which every case runs >= 3 tiles per CTA
DTYPES = {"bf16": L.DT_BF16, "f16": L.DT_F16}
U16 = {L.DT_BF16: 2.0 ** -8, L.DT_F16: 2.0 ** -11}
EPS32 = 2.0 ** -24
ONE_1 = float(np.float32(1.1))   # the kernel computes powf(1.1f, x)


@dataclass(frozen=True)
class Case:
    name: str
    cin: int                  # logical input channels of the op's input tensor
    cout: int
    k: int
    s: int
    Ho: int = 32
    Wo: int = 48
    B: int = 3
    cin_pad: int = 0          # 0: the engine's rule (64-channel chunks above 32 channels)
    in_stride: int = 0        # 0: rup(cin, 16)
    out_stride: int = 0       # 0: cout_pad
    relu: bool = True
    res: bool = False
    out_f32: bool = False
    bias_img: bool = False    # ACR_CONV_BIAS_PER_IMAGE
    pow11: bool = False       # ACR_CONV_POW11_CH0
    xpair: bool = False       # ACR_CONV_XPAIR: 64->64 on the x-paired grid, side taps = 32x32 corners
    s2x: bool = False         # ACR_CONV_S2X: input = x-paired view (2 Ho, Wo, 64) of a dense 32-channel tensor
    ext: tuple = ()           # ACR_CONV_EXTRA: nearest-upsampling shift of every extra term
    env: tuple = field(default=())   # plan-creation switches, e.g. (("ACR_B200_TMA_OUT", "1"),)

    @property
    def cinp(self):
        return self.cin_pad or (rup(self.cin, 64) if self.cin > 32 else rup(self.cin, 16))

    @property
    def coutp(self):
        return rup(self.cout, 16)

    @property
    def flags(self):
        return (self.bias_img * 1) | (self.pow11 * 2) | (self.xpair * 4) | (self.s2x * 8) | ((len(self.ext) > 0) * 16)


TMA_OUT = (("ACR_B200_TMA_OUT", "1"),)
EPI_ALL = (("ACR_B200_EPI", "2"),)

# Each row names the instance the plan heuristics give it (checked against acr_b200_conv_describe by the coverage test).
CASES = [
    # CK 16 / 32
    Case("ck16 3x3 16->64 resident, staged NB1", 16, 64, 3, 1),
    Case("ck32 1x1 32->64 resident, staged NB1", 32, 64, 1, 1, relu=False),
    Case("ck32 3x3 32->16 resident, direct N=16", 32, 16, 3, 1),
    Case("ck32 3x3 32->16 pow11, 16-bit out", 32, 16, 3, 1, relu=False, pow11=True),
    Case("ck32 3x3 96->128 streamed patch (mode 1)", 96, 128, 3, 1, cin_pad=96),
    # mode 0: streamed weights, one A box per (tap, chunk)
    Case("3x3 s2 128->256 streamed, nbuf 1", 128, 256, 3, 2),
    Case("3x3 s2 192->384 streamed, N split 2x192", 192, 384, 3, 2, Ho=16, Wo=32),
    Case("3x3 s2 256->96 streamed, nbuf 2", 256, 96, 3, 2),
    Case("3x3 s2 34(48)->384 K-padded, split, staged NB1", 34, 384, 3, 2, in_stride=48, Ho=16, Wo=32),
    Case("3x3 s2 256->64 streamed, staged NB1", 256, 64, 3, 2),
    # mode 2: resident weights
    Case("1x1 384->192 resident, nbuf 1", 384, 192, 1, 1),
    Case("1x1 64->32 resident, wider output stride", 64, 32, 1, 1, out_stride=64),
    Case("1x1 64->256 staged NB3", 64, 256, 1, 1),
    Case("1x1 64->256 + residual, staged NB3", 64, 256, 1, 1, res=True),
    Case("1x1 128->256 + residual, staged NB2", 128, 256, 1, 1, res=True),
    Case("1x1 128->256 staged NB2 (ACR_B200_EPI=2)", 128, 256, 1, 1, env=EPI_ALL),
    Case("1x1 64->512 N split 2x256, nbuf 1", 64, 512, 1, 1, relu=False),
    Case("3x3 s2 64->64 resident, staged NB1", 64, 64, 3, 2),
    Case("1x1 64->106 head, fp32 out", 64, 106, 1, 1, relu=False, out_f32=True),
    Case("1x1 64->3 cam pow11, fp32 out", 64, 3, 1, 1, relu=False, out_f32=True, pow11=True),
    Case("1x1 128->109 per-image bias, fp32 out", 128, 109, 1, 1, relu=False, out_f32=True, bias_img=True),
    Case("1x1 128->112 per-image bias, 16-bit out", 128, 112, 1, 1, bias_img=True),
    Case("1x1 64->64 + extra term >>1", 64, 64, 1, 1, ext=(1,)),
    Case("3x3 s2 64->128 + extra terms >>1 >>2 >>3", 64, 128, 3, 2, ext=(1, 2, 3)),
    # MODE_P1: one haloed box per channel chunk
    Case("3x3 34(48)->256 K-padded, P1 streamed, nbuf 1", 34, 256, 3, 1, in_stride=48),
    Case("3x3 384->384 P1, N split 2x192", 384, 384, 3, 1, Ho=16, Wo=32),
    Case("3x3 256->32 P1 streamed", 256, 32, 3, 1),
    Case("3x3 256->256 P1, N split 2x128", 256, 256, 3, 1, Ho=16, Wo=32),
    Case("3x3 128->128 + residual, P1 staged NB1", 128, 128, 3, 1, res=True),
    Case("3x3 256->256 + residual, split, staged NB1", 256, 256, 3, 1, res=True, Ho=16, Wo=32),
    Case("3x3 256->256 + residual, split, TMA store", 256, 256, 3, 1, res=True, Ho=16, Wo=32, env=TMA_OUT),
    Case("3x3 64->33(48) P1 resident, direct", 64, 33, 3, 1, relu=False),
    Case("3x3 64->64 P1 resident, staged NB1", 64, 64, 3, 1),
    Case("3x3 64->64 + residual, P1 resident, staged NB1", 64, 64, 3, 1, res=True),
    Case("3x3 64->64 + residual, P1 resident, TMA store", 64, 64, 3, 1, res=True, env=TMA_OUT),
    Case("x-paired 32->32 + residual (P1 + XPAIR)", 64, 64, 3, 1, res=True, xpair=True),
    # MODE_S2X: stride-2 conv of a dense 32-channel tensor read as x-pairs
    Case("s2x 32->256 streamed, nbuf 1", 64, 256, 3, 2, s2x=True),
    Case("s2x 32->128 streamed", 64, 128, 3, 2, s2x=True),
    Case("s2x 32->32 resident", 64, 32, 3, 2, s2x=True),
    Case("s2x 32->64 resident, staged NB1", 64, 64, 3, 2, s2x=True),
]


# ------------------------------------------------------------------------------------------------- harness
def _in_geometry(c: Case):
    """(C, H, W, pix_stride) of the op's input tensor."""
    if c.s2x:
        return 64, 2 * c.Ho, c.Wo, 64
    if c.xpair:
        return 64, c.Ho, c.Wo, 64
    return c.cin, c.Ho * c.s, c.Wo * c.s, c.in_stride or rup(c.cin, 16)


def _layout(c: Case, dt):
    """Arena regions {name: (offset, bytes)} with >= 1 KB of guard around each, the total size, and the op record."""
    Cin, Hin, Win, ins = _in_geometry(c)
    oesz = 4 if c.out_f32 else 2
    ost = c.out_stride or c.coutp
    sizes = [("x", c.B * Hin * Win * ins * 2)]
    if c.res:
        sizes.append(("res", c.B * c.Ho * c.Wo * c.coutp * 2))
    for j, sh in enumerate(c.ext):
        sizes.append((f"ext{j}", c.B * (c.Ho >> sh) * (c.Wo >> sh) * c.coutp * 2))
    if c.bias_img:
        sizes.append(("bias_img", c.B * c.coutp * 4))
    sizes.append(("out", c.B * c.Ho * c.Wo * ost * oesz))
    regions, off = {}, 1024
    for name, nbytes in sizes:
        off = rup(off, 1024)
        regions[name] = (off, nbytes)
        off += nbytes + 1024
    total = rup(off, 1024)

    op = L.Op()
    op.kind = L.OP_CONV
    op.in_[0] = ctensor(regions["x"][0], Cin, Hin, Win, ins, dt)
    n = 1
    if c.res:
        op.in_[n] = ctensor(regions["res"][0], c.cout, c.Ho, c.Wo, c.coutp, dt)
        n += 1
    for j, sh in enumerate(c.ext):
        op.in_[n] = ctensor(regions[f"ext{j}"][0], c.cout, c.Ho >> sh, c.Wo >> sh, c.coutp, dt)
        op.shift[n] = sh
        n += 1
    if c.bias_img:
        op.aux[0] = ctensor(regions["bias_img"][0], c.coutp, 1, 1, c.coutp, L.DT_F32)
    op.n_in = n
    op.out = ctensor(regions["out"][0], c.cout, c.Ho, c.Wo, ost, L.DT_F32 if c.out_f32 else dt)
    op.k, op.stride, op.relu, op.has_residual = c.k, c.s, int(c.relu), int(c.res)
    op.cin_pad, op.cout_pad = c.cinp, c.coutp
    op.shift[0] = c.flags
    return regions, total, op


def _wbytes(c: Case):
    return c.coutp * c.k * c.k * c.cinp * 2


def _tdt(dt):
    return torch.bfloat16 if dt == L.DT_BF16 else torch.float16


def _rand16(g, shape, dt, scale=1.0):
    return (torch.randn(*shape, generator=g, dtype=torch.float64) * scale).to(_tdt(dt))


def _make_data(c: Case, dt, seed):
    """Host arena (random bytes + the operands), weight blob, and the float64 operands of the reference."""
    g = torch.Generator().manual_seed(seed)
    regions, total, op = _layout(c, dt)
    arena = torch.randint(0, 256, (total,), generator=g, dtype=torch.uint8)
    Cin, Hin, Win, ins = _in_geometry(c)
    taps = c.k * c.k

    def put(name, t16):
        off, nbytes = regions[name]
        raw = t16.contiguous().view(torch.uint8).flatten()
        assert raw.numel() == nbytes
        arena[off: off + nbytes] = raw

    # input: distinct random content per image, channels beyond the logical ones zero (as the producing op leaves them)
    x = torch.zeros(c.B, Hin, Win, ins, dtype=_tdt(dt))
    x[..., :Cin] = _rand16(g, (c.B, Hin, Win, Cin), dt)
    put("x", x)
    # packed weights [cout_pad][taps][cin_pad], zero outside the logical block and where the instance does not multiply
    kin = 32 if c.s2x else Cin                                    # input channels of the convolution itself
    wp = torch.zeros(c.coutp, taps, c.cinp, dtype=torch.float64)
    wp[: c.cout, :, :Cin] = torch.randn(c.cout, taps, Cin, generator=g, dtype=torch.float64) * (2.0 / (kin * taps)) ** 0.5
    if c.xpair:     # side taps: left pair K 32..63 -> N 0..31, right pair K 0..31 -> N 32..63
        for t in range(taps):
            kx = t % 3
            if kx == 0:
                keep = torch.zeros_like(wp[:, t]); keep[:32, 32:] = wp[:32, t, 32:]; wp[:, t] = keep
            elif kx == 2:
                keep = torch.zeros_like(wp[:, t]); keep[32:, :32] = wp[32:, t, :32]; wp[:, t] = keep
    if c.s2x:       # tap (ky,kx) carries its 32 input channels at K offset 32 * (kx != 1)
        for t in range(taps):
            lo = 0 if t % 3 == 1 else 32
            keep = torch.zeros_like(wp[:, t]); keep[:, lo:lo + 32] = wp[:, t, lo:lo + 32]; wp[:, t] = keep
    w16 = wp.to(_tdt(dt))
    bias = torch.zeros(c.coutp, dtype=torch.float32)
    bias[: c.cout] = torch.randn(c.cout, generator=g) * 0.5
    blob = torch.cat([w16.view(torch.uint8).flatten(), torch.zeros(rup(_wbytes(c), 256) - _wbytes(c), dtype=torch.uint8),
                      bias.view(torch.uint8)])
    op.w_offset[0], op.w_offset[1] = 0, rup(_wbytes(c), 256)

    ops64 = {}
    xf = x.double()
    if c.s2x:       # (B, 2Ho, Wo, 64) pairs -> dense (B, 32, 2Ho, 2Wo)
        dense = xf.view(c.B, Hin, Win, 2, 32).reshape(c.B, Hin, 2 * Win, 32)
        ops64["x"] = dense.permute(0, 3, 1, 2).contiguous()
        w64 = torch.zeros(c.cout, 32, 3, 3, dtype=torch.float64)
        wu = w16.double()
        for t in range(9):
            lo = 0 if t % 3 == 1 else 32
            w64[:, :, t // 3, t % 3] = wu[: c.cout, t, lo:lo + 32]
        ops64["w"] = w64
    else:
        ops64["x"] = xf[..., :Cin].permute(0, 3, 1, 2).contiguous()
        ops64["w"] = w16.double()[: c.cout, :, :Cin].view(c.cout, c.k, c.k, Cin).permute(0, 3, 1, 2).contiguous()
    ops64["K"] = taps * kin
    if c.bias_img:
        bi = torch.zeros(c.B, c.coutp, dtype=torch.float32)
        bi[:, : c.cout] = torch.randn(c.B, c.cout, generator=g) * 0.5
        put("bias_img", bi)
        ops64["bias"] = bi[:, : c.cout].double().view(c.B, c.cout, 1, 1)
    else:
        ops64["bias"] = bias[: c.cout].double().view(1, c.cout, 1, 1)
    if c.res:
        r = torch.zeros(c.B, c.Ho, c.Wo, c.coutp, dtype=_tdt(dt))
        r[..., : c.cout] = _rand16(g, (c.B, c.Ho, c.Wo, c.cout), dt)
        put("res", r)
        ops64["res"] = r[..., : c.cout].double().permute(0, 3, 1, 2)
    ops64["ext"] = []
    for j, sh in enumerate(c.ext):
        e = torch.zeros(c.B, c.Ho >> sh, c.Wo >> sh, c.coutp, dtype=_tdt(dt))
        e[..., : c.cout] = _rand16(g, (c.B, c.Ho >> sh, c.Wo >> sh, c.cout), dt)
        put(f"ext{j}", e)
        up = e[..., : c.cout].double().permute(0, 3, 1, 2)
        ops64["ext"].append(up.repeat_interleave(1 << sh, 2).repeat_interleave(1 << sh, 3))
    # output: NaN everywhere, pad channels included
    off, nbytes = regions["out"]
    arena[off: off + nbytes] = 0xFF
    return arena, blob, op, regions, ops64


def _reference(c: Case, dt, o):
    """-> (ref, bound), float64 (B, cout, Ho, Wo)."""
    pad = 1 if c.k == 3 else 0
    conv = Fn.conv2d(o["x"], o["w"], None, c.s, pad)
    mag = Fn.conv2d(o["x"].abs(), o["w"].abs(), None, c.s, pad)
    pre = conv + o["bias"]
    amag = mag + o["bias"].abs()
    err = (o["K"] + 1) * EPS32 * amag                       # K products in fp32 + the bias add
    if c.pow11:
        p = torch.pow(ONE_1, pre[:, 0])
        e0 = p.abs() * torch.expm1(math.log(ONE_1) * err[:, 0])
        e0 = e0 + 2.0 ** -21 * (p.abs() + e0)                # powf: <= 4 ulp
        pre, amag, err = pre.clone(), amag.clone(), err.clone()
        pre[:, 0], amag[:, 0], err[:, 0] = p, p.abs(), e0
    terms = ([o["res"]] if c.res else []) + o["ext"]
    for t in terms:                                          # one fp32 rounding per added term
        pre = pre + t
        amag = amag + t.abs()
        err = err + EPS32 * amag
    ref = torch.relu(pre) if c.relu else pre
    if c.out_f32:
        return ref, err
    u = U16[dt]
    sub = 2.0 ** -25 if dt == L.DT_F16 else 0.0              # half the fp16 subnormal spacing
    return ref, u * ref.abs() + (1 + u) * err + sub


def _describe(op, B, d_arena, d_blob, dt):
    info = (C.c_int32 * len(L.CONV_INFO))()
    L.check(L.load().acr_b200_conv_describe(C.byref(op), B, d_arena.data_ptr(), d_blob.data_ptr(), dt, info, len(info)),
            "conv_describe")
    return dict(zip(L.CONV_INFO, list(info)))


def _tiles(d):
    lo, hi = d["vtiles"] // d["grid"], -(-d["vtiles"] // d["grid"])
    return lo, hi


def _row(d):
    lo, hi = _tiles(d)
    epi = ("direct", "staged", "tma-store")[d["epilogue"]]
    return (f"ck {d['ck']} MODE {d['mode']:2d} resident {d['b_resident']} nsplit {d['nsplit']} nsub {d['nsub']} "
            f"nbuf {d['nbuf']} epi {epi} nb {d['epi_nb']} SA {d['SA']} SB {d['SB']} grid {d['grid']} vtiles {d['vtiles']} "
            f"tiles/CTA {lo}-{hi}")


def _set_env(monkeypatch, c: Case, cap):
    for k, v in c.env:
        monkeypatch.setenv(k, v)
    if cap is None:
        monkeypatch.delenv(CAP_ENV, raising=False)
    else:
        monkeypatch.setenv(CAP_ENV, str(cap))


def _key(d, dt):
    """What distinguishes one compiled / scheduled form of the kernel from another."""
    return (d["ck"], "bf16" if dt == L.DT_BF16 else "f16", d["mode"], d["epilogue"], d["nbuf"], d["nsplit"] > 1)


def _check_launch(c, dt, before, after, regions, ref, bound):
    """-> worst err / bound; asserts the sentinels."""
    off_o, nb_o = regions["out"]
    ost = c.out_stride or c.coutp
    # everything but the output region is untouched: inputs first (named), then the guard bytes
    for name, (off, nbytes) in regions.items():
        if name != "out":
            assert torch.equal(after[off: off + nbytes], before[off: off + nbytes]), f"{c.name}: the {name} region changed"
    outside = torch.ones(before.numel(), dtype=torch.bool)
    for off, nbytes in regions.values():
        outside[off: off + nbytes] = False
    assert torch.equal(after[outside], before[outside]), f"{c.name}: a guard byte changed (write outside every tensor)"
    raw = after[off_o: off_o + nb_o]
    if c.out_f32:
        bits = raw.view(torch.int32).view(c.B, c.Ho, c.Wo, ost)
        val = raw.view(torch.float32).view(c.B, c.Ho, c.Wo, ost)
    else:
        bits = raw.view(torch.int16).view(c.B, c.Ho, c.Wo, ost)
        val = raw.view(_tdt(dt)).view(c.B, c.Ho, c.Wo, ost)
    assert bool((bits[..., c.cout: c.coutp] == 0).all()), f"{c.name}: pad channels {c.cout}..{c.coutp} are not +0"
    if ost > c.coutp:   # channels past cout_pad belong to other ops: still the NaN fill
        esz = 4 if c.out_f32 else 2
        px_after, px_before = raw.view(-1, ost * esz), before[off_o: off_o + nb_o].view(-1, ost * esz)
        assert torch.equal(px_after[:, c.coutp * esz:], px_before[:, c.coutp * esz:]), \
            f"{c.name}: channels past cout_pad were written"
    got = val[..., : c.cout].double().permute(0, 3, 1, 2)
    assert bool(torch.isfinite(got).all()), f"{c.name}: non-finite output (a logical channel was not written?)"
    err = (got - ref).abs()
    ratio = err / bound
    worst = float(ratio.max())
    if worst > 1.0:
        b, ch, y, x = np.unravel_index(int(ratio.argmax()), tuple(ratio.shape))
        raise AssertionError(f"{c.name}: err/bound {worst:.3g} at image {b} channel {ch} pixel ({y},{x}): got "
                             f"{float(got[b, ch, y, x]):.6g}, expected {float(ref[b, ch, y, x]):.6g}, bound "
                             f"{float(bound[b, ch, y, x]):.3g}; {int((ratio > 1).sum())} elements out of bound")
    return worst


@pytest.mark.parametrize("dtname", list(DTYPES))
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_persistent_conv(case, dtname, monkeypatch):
    dt = DTYPES[dtname]
    c = case
    torch.set_num_threads(min(32, os.cpu_count()))
    arena, blob, op, regions, ops64 = _make_data(c, dt, seed=zlib.crc32(f"{c.name} {dtname}".encode()))
    ref, bound = _reference(c, dt, ops64)
    d_arena = torch.empty_like(arena, device="cuda")
    d_blob = blob.cuda()
    outs, lines = [], []
    for cap in CAPS:
        _set_env(monkeypatch, c, cap)
        d = _describe(op, c.B, d_arena, d_blob, dt)
        d_arena.copy_(arena)
        L.check(L.load().acr_b200_run_op(C.byref(op), c.B, d_arena.data_ptr(), d_blob.data_ptr(), None, dt,
                                         torch.cuda.current_stream().cuda_stream), "run_op")
        torch.cuda.synchronize()
        after = d_arena.cpu()
        worst = _check_launch(c, dt, arena, after, regions, ref, bound)
        off, nbytes = regions["out"]
        outs.append(after[off: off + nbytes])
        lines.append(f"  cap {str(cap):>4}: {_row(d)}  worst err/bound {worst:.3f}")
        if cap == DEPTH_CAP:
            assert _tiles(d)[0] >= 3, f"{c.name}: fewer than 3 tiles per CTA at {DEPTH_CAP} CTAs ({_row(d)})"
    print(f"\n{c.name} [{dtname}, B={c.B}, {c.Ho}x{c.Wo}]\n" + "\n".join(lines))
    for cap, o in zip(CAPS[1:], outs[1:]):
        assert torch.equal(o, outs[0]), f"{c.name}: output at {cap} CTAs differs from the full grid (grid-dependent result)"


# ------------------------------------------------------------------------------------------------- coverage
MODES_REQUIRED = {0, 1, 2, 3, 17, 19, 23, 32, 34}    # 0-3 = patch / resident bits, P1, P1 + R, P1 + R + XPAIR, S2X, S2X + R


def _axes(c: Case, d):
    """Labels of the axis values a case exercises (ISSUE-level checklist of the case table)."""
    ax = {f"ck{d['ck']}", f"mode{d['mode']}"}
    epi = d["epilogue"]
    if epi == 0:
        ax.add("direct f32" if c.out_f32 else "direct 16-bit")
    elif epi == 1:
        ax.add(f"staged NB{d['epi_nb']} {'res' if c.res else 'nores'}")
    else:
        ax.add("tma store")
    ax.add(f"nsplit {d['nsplit']} nsub {d['nsub']} nbuf {d['nbuf']}")
    if c.bias_img:
        ax.add("bias per image")
    if c.pow11:
        ax.add("pow11")
    ax |= {f"extra >>{sh}" for sh in c.ext}
    return ax


AXES_REQUIRED = ({"ck16", "ck32", "ck64"} | {f"mode{m}" for m in MODES_REQUIRED}
                 | {"direct 16-bit", "direct f32", "tma store"}
                 | {f"staged NB{nb} {r}" for nb in (1, 2, 3) for r in ("res", "nores")}
                 | {"nsplit 1 nsub 64 nbuf 2", "nsplit 2 nsub 128 nbuf 2", "nsplit 2 nsub 192 nbuf 1", "nsplit 2 nsub 256 nbuf 1"}
                 | {"bias per image", "pow11", "extra >>1", "extra >>2", "extra >>3"})


def _sweep_keys(monkeypatch):
    """Instances (and axis values) the case table runs at >= 3 tiles per CTA, per dtype."""
    keys, axes = set(), {dt: set() for dt in DTYPES.values()}
    for dt in DTYPES.values():
        for c in CASES:
            _set_env(monkeypatch, c, DEPTH_CAP)
            _, total, op = _layout(c, dt)
            d_arena = torch.empty(total, dtype=torch.uint8, device="cuda")
            d_blob = torch.empty(rup(_wbytes(c), 256) + c.coutp * 4, dtype=torch.uint8, device="cuda")
            d = _describe(op, c.B, d_arena, d_blob, dt)
            for k, _ in c.env:
                monkeypatch.delenv(k)
            if _tiles(d)[0] >= 3:
                keys.add(_key(d, dt))
                axes[dt] |= _axes(c, d)
    monkeypatch.delenv(CAP_ENV)
    return keys, axes


PLANS = [   # (label, dtype, engine keyword arguments, environment at plan creation)
    ("bf16 W32", torch.bfloat16, {}, {}),
    ("fp16 W32", torch.float16, {}, {}),
    ("bf16 W48", torch.bfloat16, {"widths": "W48"}, {}),
    ("bf16 folded fuse sums", torch.bfloat16, {}, {"ACR_B200_FOLD_FUSE": "1"}),
    ("bf16 im2col stem", torch.bfloat16, {}, {"ACR_B200_STEM_FUSED": "0"}),
    ("bf16 heads only", torch.bfloat16, {"head_only": True}, {}),
]


def test_sweep_covers_every_product_instance(monkeypatch):
    """Every (CK, dtype, MODE, epilogue, nbuf, N split) a product plan launches is run by the case table above at >= 3
    tiles per CTA; if the plan heuristics move a layer to another instance, this fails instead of leaving it untested.
    With the cap unset, every plan's grid is min(virtual tiles, SMs)."""
    from acr_b200.engine import Engine
    from acr_b200.netspec import WIDTHS_W48, build_acr_spec
    from acr_b200.synth import synth_state_dict
    monkeypatch.delenv(CAP_ENV, raising=False)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    keys, axes = _sweep_keys(monkeypatch)
    for dt, got in axes.items():
        missing = AXES_REQUIRED - got
        assert not missing, f"case table misses, in {'bf16' if dt == L.DT_BF16 else 'fp16'}: {sorted(missing)}"
    sd32 = synth_state_dict(0)
    sd48 = synth_state_dict(3, spec=build_acr_spec(512, widths=WIDTHS_W48))
    missing, n_conv = {}, 0
    for label, dtype, kw, env in PLANS:
        kw = dict(kw)
        sd = sd32
        if kw.get("widths") == "W48":
            kw["widths"], sd = WIDTHS_W48, sd48
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng = Engine(sd, 2, "cuda", dtype, **kw)
        dt = eng.dt
        for i, o in enumerate(eng._cops):
            if o.kind != L.OP_CONV:
                continue
            n_conv += 1
            d = _describe(o, eng.batch, eng.arena, eng.weights, dt)
            assert d["grid"] == min(d["vtiles"], sms), (label, i, d)
            if _key(d, dt) not in keys:
                missing.setdefault(_key(d, dt), f"{label} op {i}: in {o.in_[0].C}/{o.cin_pad} -> {o.cout_pad}, k{o.k} s{o.stride}, "
                                               f"{o.out.H}x{o.out.W}, flags {o.shift[0]}; {_row(d)}")
        for k in env:
            monkeypatch.delenv(k)
        del eng
    print(f"\n{n_conv} conv launches of {len(PLANS)} plans, {len(keys)} instances in the case table at >= 3 tiles per CTA")
    assert not missing, "instances the plans launch but the case table does not run at depth:\n" + "\n".join(
        f"  {k}: {v}" for k, v in sorted(missing.items()))


# --------------------------------------------------------------------------------------------- real layers
@pytest.fixture(scope="module")
def sd():
    from acr_b200.synth import load_bn_calibration, synth_state_dict
    return synth_state_dict(0, bn_stats=load_bn_calibration(0))


def test_teacher_forced_sweep_at_seven_ctas(sd, monkeypatch):
    """Every launch of the bf16 plan at B = 1 against oracle/op_ref.py (tests/test_gpu_teacher_forced.py's sweep and
    bound), with at most 7 CTAs per conv: every layer at 64x64 and above runs >= 2 tiles per CTA (128x128: 9-10)."""
    from acr_b200.engine import Engine
    from tests.test_gpu_teacher_forced import TOL, sweep
    monkeypatch.setenv(CAP_ENV, "7")
    torch.set_num_threads(min(32, os.cpu_count()))
    gi = torch.Generator().manual_seed(123)
    image = torch.randint(0, 256, (2, 512, 512, 3), generator=gi, dtype=torch.uint8)[1:]
    eng = Engine(sd, 1, "cuda", torch.bfloat16, reuse_memory=False)
    for i, o in enumerate(eng._cops):
        if o.kind == L.OP_CONV:
            d = _describe(o, 1, eng.arena, eng.weights, eng.dt)
            assert d["grid"] == min(d["vtiles"], 7), (i, d)
            if o.out.H * o.out.W >= 64 * 64:
                assert _tiles(d)[0] >= 2, (i, _row(d))
    eng.run(image.cuda())
    torch.cuda.synchronize()
    rows = sweep(eng, sd, image, TOL[torch.bfloat16])
    worst = sorted(rows, key=lambda r: -r[2])[:5]
    print(f"\nteacher-forced sweep at 7 CTAs: {len(rows)} checks over {len(eng.recs)} launches; worst:",
          [(i, lab, f"{e:.2e}") for i, lab, e in worst])
    assert len(rows) >= len(eng.recs) - 1
    bad = [(i, lab, e) for i, lab, e in rows if not e <= TOL[torch.bfloat16]]
    assert not bad, f"{len(bad)} ops above {TOL[torch.bfloat16]:.2e}: {bad[:8]}"


def test_full_batch_256_distinct_frames(sd):
    """256 distinct frames through the bf16 plan reproduce, bit for bit, 2-frame plans run on the frames at the ends and
    the middle of the batch and at 8 more seeded positions: an image or tile index error in a deep persistent schedule
    (the 256-frame convs run up to 8192 tiles over the SMs) reads or writes another frame's data."""
    from acr_b200.engine import Engine
    B = 256
    names = ["segms", "l_center_map", "r_center_map", "l_params_maps", "r_params_maps", "l_prior_maps", "r_prior_maps",
             "pooled"]
    gi = torch.Generator().manual_seed(2026)
    frames = torch.randint(0, 256, (B, 512, 512, 3), generator=gi, dtype=torch.uint8)
    big = Engine(sd, B, "cuda")
    big.run(frames.cuda())
    torch.cuda.synchronize()
    fixed = [0, 1, 127, 128, 254, 255]
    rng = np.random.default_rng(17)
    more = sorted(int(p) for p in rng.choice(sorted(set(range(B)) - set(fixed)), 8, replace=False))
    positions = fixed + more
    small = Engine(sd, 2, "cuda", weights=big.weights)
    for pair in zip(positions[0::2], positions[1::2]):
        small.run(frames[list(pair)].contiguous().cuda())
        torch.cuda.synchronize()
        for n in names:
            C_ = big.spec.tensors[n].C
            a, b = big.view(n)[list(pair)][..., :C_], small.view(n)[..., :C_]
            assert torch.equal(a, b), f"{n}: frames {pair} of the 256-frame batch differ from a 2-frame plan"
    print(f"\n256 distinct frames: positions {positions} bit-identical to 2-frame plans")
