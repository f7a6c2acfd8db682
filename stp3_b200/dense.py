"""Host side of the dense (tensor-core) path: activation container, weight folding/packing, conv launcher.

Activations live on the device channels-last as two bf16 planes (hi, lo) with channels padded to a multiple of 64;
weights are folded (eval-mode BatchNorm -> scale/shift, reference: nn.BatchNorm eps 1e-5) and packed once per
checkpoint load into the tap-major / K-major layout stp3_conv_fwd expects (include/stp3_b200.h).
"""
import ctypes
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib

KB = 64  # channels per K block


def pad_to(c: int, m: int = KB) -> int:
    return (c + m - 1) // m * m


def out_tile(c: int) -> int:
    """Padded output-channel tile of the conv kernel (UMMA N): 64, 128 or 256."""
    for bn in (64, 128, 256):
        if c <= bn:
            return bn
    raise ValueError(f"{c} output channels: split the convolution (max 256 per launch)")


@dataclass
class HL:
    """(B, T, H, W, Cp) fp32 tensor carried as bf16 hi/lo planes; `c` = number of real channels."""
    hi: torch.Tensor
    lo: torch.Tensor
    c: int

    @property
    def shape(self):
        return self.hi.shape

    @staticmethod
    def empty(B, T, H, W, c, device, cp=None):
        cp = cp or pad_to(c)
        return HL(torch.empty((B, T, H, W, cp), dtype=torch.bfloat16, device=device),
                  torch.empty((B, T, H, W, cp), dtype=torch.bfloat16, device=device), c)

    @staticmethod
    def zeros(B, T, H, W, c, device, cp=None):
        cp = cp or pad_to(c)
        return HL(torch.zeros((B, T, H, W, cp), dtype=torch.bfloat16, device=device),
                  torch.zeros((B, T, H, W, cp), dtype=torch.bfloat16, device=device), c)


def split_hilo(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return hi, lo


def fold_bn(weight: torch.Tensor, bn: Optional[torch.nn.modules.batchnorm._BatchNorm], conv_bias=None):
    """conv (no bias) -> eval BatchNorm  ==  conv with w*s and bias (beta - mean*s), s = gamma/sqrt(var+eps)."""
    cout = weight.shape[0]
    w = weight.detach().float()
    b = conv_bias.detach().float() if conv_bias is not None else torch.zeros(cout, device=w.device)
    if bn is not None:
        s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
        w = w * s.view(-1, *([1] * (w.dim() - 1)))
        b = (b - bn.running_mean.detach().float()) * s + bn.bias.detach().float()
    return w, b


@dataclass
class PackedConv:
    w: torch.Tensor            # [ntaps][cin_p/64][2][bn][64] bf16
    bias: torch.Tensor         # [bn] fp32
    taps: List[Tuple[int, int, int]]
    cin_p: int
    bn: int
    cout: int
    stride: int
    k_lo: int = 0              # input channels [k_lo, k_hi) of the window carry weights (multiples of 16)
    k_hi: int = 0
    uid: int = 0               # identity of this packing for the autotune cache (a data_ptr can be reused after a repack)


_PACK_COUNTER = 0


def pack_conv(weight: torch.Tensor, bias: torch.Tensor, *, stride: int = 1, dilation: int = 1,
              padding: Optional[int] = None, causal_time: bool = True, cin_p: Optional[int] = None,
              bn: Optional[int] = None, prune_extent: Optional[Tuple[int, int]] = None,
              in_layout: Optional[Sequence[Tuple[int, int, int]]] = None) -> PackedConv:
    """weight: (Cout, Cin, kh, kw) or (Cout, Cin, kt, kh, kw), already BN-folded; bias (Cout).
    Taps are (dt, dy, dx) input offsets: dy = ky*dilation - padding (padding defaults to 'same'); for 3-D kernels
    dt = kt_index - (kt - 1) (causal: the reference pads time on the left only, temporal.py:256-262)."""
    if weight.dim() == 4:
        weight = weight.unsqueeze(2)
    cout, cin, kt, kh, kw = weight.shape
    pad_h = padding if padding is not None else (kh - 1) * dilation // 2
    pad_w = padding if padding is not None else (kw - 1) * dilation // 2
    # in_layout: [(first logical input channel, count, physical channel offset)] -- where each group of the
    # convolution's input channels lives inside the (padded / concatenated) physical input window
    in_layout = list(in_layout) if in_layout is not None else [(0, cin, 0)]
    cin_p = cin_p or pad_to(max(off + n for _, n, off in in_layout))
    bn = bn or out_tile(cout)
    dev = weight.device
    taps, mats = [], []
    for it in range(kt):
        for ix in range(kw):              # dy innermost: runs of taps whose dy advance by the stride share one
            # activation load (stride 1: dy, dy+1, dy+2; stride 2: the even rows of the kernel, then the odd ones)
            for iy in (list(range(0, kh, 2)) + list(range(1, kh, 2)) if stride == 2 else range(kh)):
                dy, dx = iy * dilation - pad_h, ix * dilation - pad_w
                if prune_extent is not None and stride == 1:
                    # a tap whose shift exceeds the image reads only zero padding for every output pixel
                    H, W = prune_extent
                    if abs(dy) >= H or abs(dx) >= W:
                        continue
                taps.append((it - (kt - 1) if causal_time else it, dy, dx))
                m = torch.zeros((bn, cin_p), dtype=torch.float32, device=dev)
                for src, n, off in in_layout:
                    m[:cout, off:off + n] = weight[:, src:src + n, it, iy, ix]
                mats.append(m)
    w = torch.stack(mats)                                            # (ntaps, bn, cin_p)
    hi, lo = split_hilo(w)
    nt = len(taps)
    kbs = cin_p // KB
    packed = torch.stack([hi.view(nt, bn, kbs, KB), lo.view(nt, bn, kbs, KB)], dim=0)   # (2, nt, bn, kbs, 64)
    packed = packed.permute(1, 3, 0, 2, 4).contiguous()              # (nt, kbs, 2, bn, 64)
    b = torch.zeros(bn, dtype=torch.float32, device=dev)
    b[:cout] = bias
    k_lo = min(off for _, _, off in in_layout) // 16 * 16
    k_hi = (max(off + n for _, n, off in in_layout) + 15) // 16 * 16
    if not (k_lo < KB and k_hi > cin_p - KB):          # the kernel trims only the first / last 64-channel block
        k_lo, k_hi = 0, cin_p
    global _PACK_COUNTER
    _PACK_COUNTER += 1
    return PackedConv(packed, b, taps, cin_p, bn, cout, stride, k_lo, k_hi, _PACK_COUNTER)


# ------------------------------------------------------------------------------------------------ autotuner
# The conv kernel has two tiling knobs (sub-tiles per CTA tile -- or a 16x16 tile shared by a CTA pair through
# tcgen05.mma.cta_group::2, n_sub = 3 -- and sharing one activation load between the dy taps of a 3x3).  2-D layers over
# every frame also get the linear tiling (n_sub 4 / 5 = 128 / 256 consecutive output pixels per CTA / CTA pair, one
# im2col load per tap; no pixels of padding on small maps, and a 256-column layer runs as one launch).  Which
# combination wins depends on the layer (K depth, N width, image size, whether the weights are
# smem-resident), so the first eager call of every (layer, shape) times the candidates back to back and the winner is
# cached; CUDA-graph capture then records the tuned launches.  STP3_CONV_AUTOTUNE=0 disables it (kernel heuristics).
import os as _os

_TUNED = {}
_AUTOTUNE = _os.environ.get("STP3_CONV_AUTOTUNE", "1") != "0"
_TUNE_PAIR = _os.environ.get("STP3_CONV_PAIR", "1") != "0"
TUNE_LOG = []      # (description, {config: ms}) for reports


def _tune(key, desc, launch, groupable, ntaps=1, bn=0, linear=False):
    cands = [(1, 1), (2, 1)] + ([(1, 3), (2, 3)] if groupable else [])
    if _TUNE_PAIR:
        cands += [(3, 1)] + ([(3, 3)] if groupable else [])
    if linear:          # group 3 / 1 only picks the tap order (the same as the 2-D tiling with that group)
        for ns in ((4, 5) if _TUNE_PAIR else (4,)):
            cands += [(ns, 1)] + ([(ns, 3)] if groupable else [])
    if ntaps > 1:       # weights streamed through the ring instead of resident: more activation stages in flight
        cands += [(ns, g + 4) for ns, g in cands if ns != 1]
    if bn == 64:        # stacked [W_hi; W_lo] operand: two MMAs per product instead of three
        cands += [(ns, g + 8) for ns, g in cands]
    times = {}
    for ns, g in cands:
        launch(ns, g)                                   # warm (descriptor / attribute setup)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(4):
            launch(ns, g)
        b.record()
        b.synchronize()
        times[(ns, g)] = a.elapsed_time(b) / 4
    best = min(times, key=times.get)
    _TUNED[key] = best
    TUNE_LOG.append((desc, times))
    return best


def conv(x: HL, pc: PackedConv, *, cin_off: int = 0, out: Optional[HL] = None, out_coff: int = 0, relu: bool = False,
         img_bias: Optional[torch.Tensor] = None, residual: Optional[HL] = None, res_coff: int = 0,
         res_after_act: bool = False, out_f32: Optional[torch.Tensor] = None, n_valid: int = 0, sigmoid: bool = False,
         out_hw: Optional[Tuple[int, int]] = None, n_store: int = 0, frames: Optional[Tuple[int, int]] = None,
         head: Optional[dict] = None, store: bool = True, tune: Optional[Tuple[int, int]] = None,
         col_sums: Optional[torch.Tensor] = None, out2: Optional[HL] = None, out2_coff: int = 0, n_store2: int = 0,
         relu2: bool = False, out_f32_nhwc: bool = False) -> Optional[HL]:
    """y = act(conv(x[..., cin_off:cin_off+cin]) + bias [+ residual]) written into out[..., out_coff:...]; when
    img_bias (n_img, bn) is given it REPLACES the convolution's bias vector (build it with bias_table()).
    out2 (bn = 128 layers, n_store <= 64): output columns [64, 64+n_store2) go to out2[..., out2_coff:...] with activation
    relu2 -- two 64-column convolutions of the same input in one launch.
    col_sums (B*T, 64) fp32 (bn = 64 layers): receives the per-image sums over pixels of the activated output.
    tune = (n_sub, group) forces a tiling (n_sub 3 = CTA pair, 4 / 5 = linear tiling per CTA / CTA pair; group +4 =
    streamed weights, +8 = stacked hi/lo weight operand) instead of the autotuned one."""
    B, T_total, H, W, cs = x.hi.shape
    t0, T = frames if frames is not None else (0, T_total)      # process frames [t0, t0+T) of every sample
    Ho, Wo = out_hw if out_hw is not None else ((H + pc.stride - 1) // pc.stride, (W + pc.stride - 1) // pc.stride)
    d = _lib.ConvDesc()
    d.B, d.T, d.H, d.W = B, T, H, W
    d.T_total, d.t0 = T_total, t0
    d.in_cstride, d.cin_off, d.cin = cs, cin_off, pc.cin_p
    d.Ho, d.Wo, d.stride = Ho, Wo, pc.stride
    d.ntaps = len(pc.taps)
    for i, (dt, dy, dx) in enumerate(pc.taps):
        d.taps[i][0], d.taps[i][1], d.taps[i][2] = dt, dy, dx
    d.bn = pc.bn
    d.n_cols = pc.cout              # weight rows / bias entries beyond cout are zero padding
    d.k_lo, d.k_hi = pc.k_lo, pc.k_hi
    if out is None and out_f32 is None and store:
        out = HL.empty(B, T, Ho, Wo, pc.cout, x.hi.device, cp=pc.bn)
    hd = None
    if head is not None:
        # fused 1x1 head: dict(w (KO,bn) f32, b (KO) f32, outs=[(tensor (n_img,k,Ho,Wo) f32, channel)], sigmoid_mask)
        hd = _lib.ConvHead()
        hd.n_out = len(head["outs"])
        assert head["w"].shape == (hd.n_out, pc.bn) and head["w"].is_contiguous() and head["b"].numel() == hd.n_out
        hd.w, hd.b = head["w"].data_ptr(), head["b"].data_ptr()
        for k, (t, ch) in enumerate(head["outs"]):
            assert t.dtype == torch.float32 and t.is_contiguous() and t.shape[0] == B * T and t.shape[2:] == (Ho, Wo)
            hd.out[k] = t.data_ptr() + ch * Ho * Wo * 4
            hd.img_stride[k] = t.shape[1] * Ho * Wo
        hd.sigmoid_mask = int(head.get("sigmoid_mask", 0))
    if out is not None:
        assert out.hi.shape[:4] == (B, T, Ho, Wo), (out.hi.shape, (B, T, Ho, Wo))
        d.out_cstride, d.out_coff, d.n_store = out.hi.shape[-1], out_coff, n_store
    d.relu = int(relu)
    if residual is not None:
        d.res_mode = 2 if res_after_act else 1
        d.res_cstride, d.res_coff = residual.hi.shape[-1], res_coff
        assert residual.hi.shape[:4] == (B, T, Ho, Wo)
    d.n_valid, d.sigmoid = n_valid, int(sigmoid)
    d.f32_layout = int(out_f32_nhwc)        # out_f32 (B*T, Ho, Wo, n_valid) instead of (B*T, n_valid, Ho, Wo)
    if out2 is not None:
        assert pc.bn == 128 and out is not None and out2.hi.shape[:4] == (B, T, Ho, Wo)
        d.y2_hi, d.y2_lo = out2.hi.data_ptr(), out2.lo.data_ptr()
        d.out2_cstride, d.out2_coff, d.n_store2, d.relu2 = out2.hi.shape[-1], out2_coff, n_store2, int(relu2)
    scratch = None
    if col_sums is not None:
        assert pc.bn == 64 and col_sums.shape == (B * T, 64) and col_sums.dtype == torch.float32 and col_sums.is_contiguous()
        nbytes = _lib.lib().stp3_conv_col_sums_scratch_bytes(B * T, 64)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.hi.device)
        d.col_sums, d.col_sums_scratch, d.col_sums_scratch_bytes = col_sums.data_ptr(), scratch.data_ptr(), nbytes
    if img_bias is not None:
        assert img_bias.shape == (B * T, pc.bn) and img_bias.dtype == torch.float32 and img_bias.is_contiguous()
    dev = x.hi.device
    ptr = lambda t: t.data_ptr() if t is not None else None

    def launch(n_sub=0, group=0):
        d.tune_n_sub, d.tune_group = n_sub, group
        with torch.cuda.device(dev):
            code = _lib.lib().stp3_conv_fwd(
                ctypes.byref(d), x.hi.data_ptr(), x.lo.data_ptr(), pc.w.data_ptr(), pc.bias.data_ptr(), ptr(img_bias),
                ptr(residual.hi if residual is not None else None), ptr(residual.lo if residual is not None else None),
                ptr(out.hi if out is not None else None), ptr(out.lo if out is not None else None), ptr(out_f32),
                ctypes.byref(hd) if hd is not None else None, torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(code, "stp3_conv_fwd")

    key = (pc.uid, B, T, H, W, cs, cin_off, Ho, Wo, t0, int(relu), residual is not None, out_f32 is not None,
           hd is not None, out2 is not None)
    cfg = tune if tune is not None else _TUNED.get(key)
    if cfg is None and _AUTOTUNE and not torch.cuda.is_current_stream_capturing():
        taps = pc.taps
        groupable = any(taps[i + 1][0] == taps[i][0] and taps[i + 1][2] == taps[i][2] and
                        taps[i + 1][1] == taps[i][1] + pc.stride for i in range(len(taps) - 1))
        desc = f"{len(taps)}tap cin{pc.cin_p} bn{pc.bn} s{pc.stride} {B * T}x{Ho}x{Wo}"
        # the tuner launches the layer many times: an output that aliases an input would be corrupted silently
        ins = {x.hi.data_ptr(), x.lo.data_ptr()} | ({residual.hi.data_ptr(), residual.lo.data_ptr()} if residual is not None else set())
        outs = {t.data_ptr() for t in ((out.hi, out.lo) if out is not None else ()) + ((out2.hi, out2.lo) if out2 is not None else ())}
        assert not (ins & outs), "stp3_b200.dense.conv: output aliases an input (in-place convolution is not supported)"
        linear = (all(t[0] == 0 for t in taps) and (t0, T) == (0, T_total) and col_sums is None and hd is None and
                  img_bias is None and out_f32 is None)
        cfg = _tune(key, desc, launch, groupable, len(taps), pc.bn, linear)
    launch(*(cfg or (0, 0)))
    return out


@dataclass
class PackedAspp:
    w: torch.Tensor            # bf16 rows of 64: [tap/K blocks ...][projection blocks ...], each [hi 128][lo 128]
    br_bias: torch.Tensor      # (n_br, 128) fp32
    proj_bias: torch.Tensor    # (128,) fp32
    taps: List[List[Tuple[int, int]]]
    cin_p: int


def pack_aspp(branches, proj_w: torch.Tensor, proj_b: torch.Tensor) -> PackedAspp:
    """branches: [(weight (128, Cin, kh, kw) BN-folded, bias (128), dilation)]; proj_w (<= 128, n_br * 128) BN-folded
    (fewer than 128 output rows are zero-padded).  Layout of stp3_aspp_fused_fwd (include/stp3_b200.h)."""
    h = 128
    if proj_w.shape[0] < h:
        pw = torch.zeros((h, proj_w.shape[1]), dtype=proj_w.dtype, device=proj_w.device)
        pw[:proj_w.shape[0]] = proj_w
        pb = torch.zeros(h, dtype=proj_b.dtype, device=proj_b.device)
        pb[:proj_b.shape[0]] = proj_b
        proj_w, proj_b = pw, pb
    cin = branches[0][0].shape[1]
    cin_p = pad_to(cin)
    kbs = cin_p // KB
    dev = proj_w.device
    blocks, taps_all, biases = [], [], []
    for w, b, dil in branches:
        assert w.shape[0] == h and w.shape[1] == cin
        kh, kw = w.shape[2:]
        taps = []
        for iy in range(kh):
            for ix in range(kw):
                dy, dx = (iy - (kh - 1) // 2) * dil, (ix - (kw - 1) // 2) * dil
                taps.append((dy, dx))
                m = torch.zeros((h, cin_p), dtype=torch.float32, device=dev)
                m[:, :cin] = w[:, :, iy, ix]
                for kb in range(kbs):
                    blocks.append(m[:, kb * KB:(kb + 1) * KB])
        taps_all.append(taps)
        biases.append(b)
    for i in range(len(branches)):
        for kb2 in range(2):
            blocks.append(proj_w[:, i * h + kb2 * KB: i * h + (kb2 + 1) * KB])
    m = torch.stack(blocks).float()                                   # (n_blocks, 128, 64)
    hi, lo = split_hilo(m)
    packed = torch.stack([hi, lo], dim=1).contiguous()                # (n_blocks, 2, 128, 64)
    return PackedAspp(packed, torch.stack(biases).float().contiguous(), proj_b.float().contiguous(), taps_all, cin_p)


def aspp_fused(x: HL, pa: PackedAspp, img_bias: torch.Tensor, out: Optional[HL] = None, out_coff: int = 0,
               relu: bool = True, n_store: int = 128, c_out: Optional[int] = None) -> HL:
    """y = [relu](project(cat_b relu(branch_b(x))) + img_bias): stp3_aspp_fused_fwd.  n_store = 64: only the first 64
    output channels exist (c_out of them real)."""
    B, T, H, W, cs = x.hi.shape
    if out is None:
        out = HL.empty(B, T, H, W, c_out or n_store, x.hi.device, cp=n_store)
    assert img_bias.shape == (B * T, 128) and img_bias.dtype == torch.float32 and img_bias.is_contiguous()
    d = _lib.AsppDesc()
    d.B, d.T, d.H, d.W, d.in_cstride, d.cin = B, T, H, W, cs, pa.cin_p
    d.n_br = len(pa.taps)
    for b, taps in enumerate(pa.taps):
        d.n_taps[b] = len(taps)
        for i, (dy, dx) in enumerate(taps):
            d.taps[b][i][0], d.taps[b][i][1] = dy, dx
    d.out_cstride, d.out_coff = out.hi.shape[-1], out_coff
    d.no_relu, d.n_store = int(not relu), n_store
    with torch.cuda.device(x.hi.device):
        code = _lib.lib().stp3_aspp_fused_fwd(ctypes.byref(d), x.hi.data_ptr(), x.lo.data_ptr(), pa.w.data_ptr(),
                                              pa.br_bias.data_ptr(), img_bias.data_ptr(), out.hi.data_ptr(),
                                              out.lo.data_ptr(), torch.cuda.current_stream(x.hi.device).cuda_stream)
    _lib.check(code, "stp3_aspp_fused_fwd")
    return out


@dataclass
class PackedBlockTail:
    w: torch.Tensor                 # (n_blocks, 2, 128, 64) bf16
    chains: list                    # [(src, cin_off, taps [(dt,dy,dx)], n_mma, tmem_col, k_lo, k_hi)]
    res: Optional[tuple]            # the projection chain or None (identity residual)
    piece_col: List[int]


def _pair_rows(m: torch.Tensor) -> torch.Tensor:
    """(N, 64) weight rows of an N-wide chain -> (128, 64): row n of the first / second half of N at row n / 64 + n - N/2
    (each CTA of a pair loads 64 rows and multiplies its N/2)."""
    n = m.shape[0]
    out = torch.zeros((128, KB), dtype=torch.float32, device=m.device)
    out[:n // 2] = m[:n // 2]
    out[64:64 + n - n // 2] = m[n // 2:]
    return out


def pack_block_tail(chains, agg_w: torch.Tensor, res_w: Optional[torch.Tensor], piece_col) -> PackedBlockTail:
    """chains: [(src, cin_off, weight (cout, cin, kt, kh, kw) BN-folded, k_off, n_mma, tmem_col)] -- cin input channels of
    the chain sit at channels [k_off, k_off + cin) of its 64-channel K block; agg_w (64, 128) aggregation weights in P
    order; res_w (64, cs) projection weights or None."""
    dev = agg_w.device
    blocks, desc = [], []
    for src, cin_off, w, k_off, n_mma, tmem_col in chains:
        cout, cin, kt, kh, kw = w.shape
        assert cout <= n_mma and k_off + cin <= KB
        taps = []
        for it in range(kt):
            for ix in range(kw):
                for iy in range(kh):
                    taps.append((it - (kt - 1), iy - (kh - 1) // 2, ix - (kw - 1) // 2))
                    m = torch.zeros((n_mma, KB), dtype=torch.float32, device=dev)
                    m[:cout, k_off:k_off + cin] = w[:, :, it, iy, ix]
                    blocks.append(_pair_rows(m))
        desc.append((src, cin_off, taps, n_mma, tmem_col, k_off // 16 * 16, (k_off + cin + 15) // 16 * 16))
    for kb2 in range(2):
        blocks.append(_pair_rows(agg_w[:, kb2 * KB:(kb2 + 1) * KB].float()))
    res = None
    if res_w is not None:
        cs = res_w.shape[1]
        m = torch.zeros((64, KB), dtype=torch.float32, device=dev)
        m[:res_w.shape[0], :cs] = res_w
        blocks.append(_pair_rows(m))
        res = (1, 0, [(0, 0, 0)], 64, 0, 0, (cs + 15) // 16 * 16)
    hi, lo = split_hilo(torch.stack(blocks))
    return PackedBlockTail(torch.stack([hi, lo], dim=1).contiguous(), desc, res, list(piece_col))


def block_tail(mid: HL, x: HL, pb: PackedBlockTail, hid_bias: torch.Tensor, img_bias: torch.Tensor,
               res_bias: Optional[torch.Tensor], col_sums: Optional[torch.Tensor] = None) -> HL:
    """stp3_block_fused_fwd: the paths, the aggregation convolution and the residual of a TemporalBlock in one kernel."""
    B, T, H, W, _ = x.hi.shape
    out = HL.empty(B, T, H, W, 64, x.hi.device, cp=64)
    d = _lib.BlockDesc()
    d.B, d.T, d.H, d.W = B, T, H, W
    d.mid_cstride, d.x_cstride, d.out_cstride = mid.hi.shape[-1], x.hi.shape[-1], 64

    def fill(dst, c):
        src, cin_off, taps, n_mma, tmem_col, k_lo, k_hi = c
        dst.src, dst.cin_off, dst.n_taps, dst.n_mma, dst.tmem_col, dst.k_lo, dst.k_hi = src, cin_off, len(taps), n_mma, tmem_col, k_lo, k_hi
        for i, (dt, dy, dx) in enumerate(taps):
            dst.taps[i][0], dst.taps[i][1], dst.taps[i][2] = dt, dy, dx
    d.n_chain = len(pb.chains)
    for i, c in enumerate(pb.chains):
        fill(d.chain[i], c)
    d.has_res_proj = int(pb.res is not None)
    if pb.res is not None:
        fill(d.res, pb.res)
    for i, v in enumerate(pb.piece_col):
        d.piece_col[i] = v
    n_img = B * T
    assert hid_bias.shape == (n_img, 128) and img_bias.shape == (n_img, 64) and hid_bias.is_contiguous() and img_bias.is_contiguous()
    assert (res_bias is None) == (pb.res is None)
    scratch, nbytes = None, 0
    if col_sums is not None:
        assert col_sums.shape == (n_img, 64) and col_sums.dtype == torch.float32 and col_sums.is_contiguous()
        nbytes = _lib.lib().stp3_block_fused_scratch_bytes(n_img)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.hi.device)
    ptr = lambda t: t.data_ptr() if t is not None else None
    with torch.cuda.device(x.hi.device):
        code = _lib.lib().stp3_block_fused_fwd(
            ctypes.byref(d), mid.hi.data_ptr(), mid.lo.data_ptr(), x.hi.data_ptr(), x.lo.data_ptr(), pb.w.data_ptr(),
            hid_bias.data_ptr(), img_bias.data_ptr(), ptr(res_bias), out.hi.data_ptr(), out.lo.data_ptr(), ptr(col_sums),
            ptr(scratch), nbytes, torch.cuda.current_stream(x.hi.device).cuda_stream)
    _lib.check(code, "stp3_block_fused_fwd")
    return out


def bias_table(pc: PackedConv, n_img: int) -> torch.Tensor:
    """(n_img, bn) per-image bias initialised with the convolution's own bias; the spatially constant branches are
    accumulated on top (pool_bias / small_linear with accumulate=True)."""
    return pc.bias.unsqueeze(0).expand(n_img, -1).contiguous()


# ------------------------------------------------------------------------------------------------ aux kernels
def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def from_f32(x: torch.Tensor, channels_last: bool = False, cp: Optional[int] = None) -> HL:
    """x (B,T,C,H,W) [or (B,T,H,W,C)] fp32 on the device -> HL (CUDA transpose + hi/lo split)."""
    if not x.is_cuda:
        raise RuntimeError("stp3_b200 dense ops run on CUDA tensors only (there is no CPU path)")
    x = x.detach().float().contiguous()
    if channels_last:
        B, T, H, W, C = x.shape
    else:
        B, T, C, H, W = x.shape
    out = HL.empty(B, T, H, W, C, x.device, cp=cp)
    with torch.cuda.device(x.device):
        code = _lib.lib().stp3_f32_to_hilo(x.data_ptr(), int(channels_last), B * T, C, H, W, out.hi.shape[-1],
                                           out.hi.data_ptr(), out.lo.data_ptr(), _stream(x.device))
    _lib.check(code, "stp3_f32_to_hilo")
    return out


def to_f32(x: HL, c_off: int = 0, c: Optional[int] = None) -> torch.Tensor:
    """HL -> (B,T,C,H,W) fp32 (the reference's layout)."""
    B, T, H, W, cs = x.hi.shape
    c = c if c is not None else x.c
    out = torch.empty((B, T, c, H, W), dtype=torch.float32, device=x.hi.device)
    with torch.cuda.device(x.hi.device):
        code = _lib.lib().stp3_hilo_to_f32(x.hi.data_ptr(), x.lo.data_ptr(), B * T, H, W, cs, c_off, c, out.data_ptr(),
                                           _stream(x.hi.device))
    _lib.check(code, "stp3_hilo_to_f32")
    return out


def spatial_sum(x: HL) -> torch.Tensor:
    """(B*T, cstride) fp32 sums over the H*W pixels of every image."""
    B, T, H, W, cs = x.hi.shape
    out = torch.empty((B * T, cs), dtype=torch.float32, device=x.hi.device)
    with torch.cuda.device(x.hi.device):
        code = _lib.lib().stp3_spatial_sum(x.hi.data_ptr(), x.lo.data_ptr(), B * T, H * W, cs, out.data_ptr(),
                                           _stream(x.hi.device))
    _lib.check(code, "stp3_spatial_sum")
    return out


def pool_bias(sums: torch.Tensor, T: int, C: int, hw: int, temporal: bool, W1, b1, W2, out: torch.Tensor,
              accumulate: bool, const: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None):
    """out[img, :CO] = (out | bias | 0) + W2 relu(W1 mean + b1): a spatially constant branch as a per-image bias (see
    header).  const (n_img, n_const): values of the trailing spatially constant input channels (not part of sums)."""
    n_img = sums.shape[0]
    R, CO = W1.shape[0], W2.shape[0]
    nc = 0 if const is None else const.shape[1]
    assert W1.shape == (R, C) and W2.shape == (CO, R) and out.shape[0] == n_img and C - nc <= sums.shape[1]
    for t in (sums, W1, b1, W2, out) + ((const,) if nc else ()) + ((bias,) if bias is not None else ()):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.is_cuda
    assert bias is None or bias.numel() >= CO
    with torch.cuda.device(sums.device):
        code = _lib.lib().stp3_pool_bias(sums.data_ptr(), sums.shape[1], n_img, T, C, 1.0 / hw, int(temporal),
                                         const.data_ptr() if nc else None, nc,
                                         W1.data_ptr(), b1.data_ptr(), R, W2.data_ptr(), CO,
                                         bias.data_ptr() if bias is not None else None, out.data_ptr(),
                                         out.shape[1], int(accumulate), _stream(sums.device))
    _lib.check(code, "stp3_pool_bias")


def small_linear(x: torch.Tensor, W: torch.Tensor, out: torch.Tensor, accumulate: bool,
                 bias: Optional[torch.Tensor] = None):
    """out[n, :co] = (out | bias | 0) + W x[n]."""
    n, ci = x.shape
    co = W.shape[0]
    assert W.shape == (co, ci) and out.shape[0] == n
    for t in (x, W, out) + ((bias,) if bias is not None else ()):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.is_cuda
    assert bias is None or bias.numel() >= co
    with torch.cuda.device(x.device):
        code = _lib.lib().stp3_small_linear(x.data_ptr(), W.data_ptr(), n, ci, co,
                                            bias.data_ptr() if bias is not None else None, out.data_ptr(),
                                            out.shape[1], int(accumulate), _stream(x.device))
    _lib.check(code, "stp3_small_linear")


def upsample2x_add(x: HL, skip: Optional[HL], c: int, skip_coff: int = 0, out: Optional[HL] = None,
                   out_coff: int = 0) -> HL:
    """out[..., out_coff:out_coff+c] = bilinear x2 (align_corners=False) of x[..., :c] (+ skip[..., skip_coff:+c])."""
    B, T, h, w, xs = x.hi.shape
    if skip is not None:
        assert skip.hi.shape[:4] == (B, T, 2 * h, 2 * w)
    if out is None:
        out = HL.empty(B, T, 2 * h, 2 * w, c, x.hi.device, cp=c)
    assert out.hi.shape[:4] == (B, T, 2 * h, 2 * w)
    ptr = lambda t: t.data_ptr() if t is not None else None
    with torch.cuda.device(x.hi.device):
        code = _lib.lib().stp3_upsample2x_add(
            x.hi.data_ptr(), x.lo.data_ptr(), B * T, h, w, xs, ptr(skip.hi if skip else None),
            ptr(skip.lo if skip else None), skip.hi.shape[-1] if skip else 0, skip_coff, out.hi.data_ptr(),
            out.lo.data_ptr(), out.hi.shape[-1], out_coff, c, _stream(x.hi.device))
    _lib.check(code, "stp3_upsample2x_add")
    return out
