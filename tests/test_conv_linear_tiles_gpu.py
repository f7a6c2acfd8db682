"""GPU tests of the linear conv tiling (tune n_sub 4 = 128 consecutive output pixels per CTA, 5 = 256 per CTA pair,
one im2col TMA load per tap): every decoder layer at its real shape against the fp64 convolution and, bit for bit,
against the 2-D CTA-pair tiling that issues the taps in the same order; tiles that cross images, the last partial
tile, and the layers the linear tiling refuses."""
import pytest
import torch
import torch.nn.functional as F

from stp3_b200 import dense
from tests.test_conv_gpu import check, rnd

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_IMG = 12          # B * S of the perceive benchmark (4 samples x 3 frames)


def to_hl_dev(x, cp=None):
    """x (B, T, C, H, W) fp32 on the device -> HL."""
    B, T, C, H, W = x.shape
    xp = torch.zeros(B, T, H, W, cp or dense.pad_to(C), device=DEV)
    xp[..., :C] = x.permute(0, 1, 3, 4, 2)
    hi, lo = dense.split_hilo(xp)
    return dense.HL(hi.contiguous(), lo.contiguous(), C)


def hl_f32(h, c):
    return (h.hi.float() + h.lo.float())[..., :c].permute(0, 1, 4, 2, 3)


def ref_conv(x, w, b, stride):
    B, T, C, H, W = x.shape
    y = F.conv2d(x.reshape(B * T, C, H, W).double(), w.double(), b.double(), stride=stride,
                 padding=(w.shape[-1] - 1) // 2)
    return y.view(B, T, *y.shape[1:])


def layer(cin, cout, k, stride, hw, seed, n_img=N_IMG):
    x = rnd(1, n_img, cin, hw, hw, seed=seed).to(DEV)
    w = rnd(cout, cin, k, k, seed=seed + 1, scale=(cin * k * k) ** -0.5).to(DEV)
    b = rnd(cout, seed=seed + 2).to(DEV)
    return x, w, b, dense.pack_conv(w, b, stride=stride)


def groupable(pc):
    t = pc.taps
    return any(t[i + 1][0] == t[i][0] and t[i + 1][2] == t[i][2] and t[i + 1][1] == t[i][1] + pc.stride
               for i in range(len(t) - 1))


# the decoder's convolutions (models/decoder.py) at 200x200 BEV, 12 images; 25 -> 13 is an odd stride-2 output
DECODER_LAYERS = [
    (64, 64, 7, 2, 200),      # first_conv 7x7 s2 -> 100^2
    (64, 64, 3, 1, 100),      # layer1
    (64, 128, 3, 2, 100),     # layer2.0.c1 -> 50^2
    (64, 128, 1, 2, 100),     # layer2.0.ds
    (128, 128, 3, 1, 50),     # layer2 c2 / c1
    (128, 256, 3, 2, 50),     # layer3.0.c1 -> 25^2, 256 columns in one launch
    (128, 256, 1, 2, 50),     # layer3.0.ds
    (256, 256, 3, 1, 25),     # layer3 c2 / c1
    (256, 256, 3, 2, 25),     # 25 -> 13
]


@pytest.mark.parametrize("mode", [4, 5])
@pytest.mark.parametrize("cin,cout,k,stride,hw", DECODER_LAYERS)
def test_decoder_layer_linear_matches_fp64_and_2d(mode, cin, cout, k, stride, hw):
    x, w, b, pc = layer(cin, cout, k, stride, hw, seed=100 + k + cin)
    xh = to_hl_dev(x)
    g = 3 if groupable(pc) else 1
    stacks = [0, 8] if pc.bn == 64 and k > 1 else [0]
    ref = F.relu(ref_conv(x, w, b, stride))
    for st in stacks:
        y_lin = dense.conv(xh, pc, relu=True, tune=(mode, g + st))
        y_2d = dense.conv(xh, pc, relu=True, tune=(3, g + st))
        torch.cuda.synchronize()
        check(hl_f32(y_lin, cout), ref)
        # same taps in the same order per pixel: the same fp32 sums
        assert torch.equal(y_lin.hi, y_2d.hi) and torch.equal(y_lin.lo, y_2d.lo), (mode, st)


@pytest.mark.parametrize("mode", [4, 5])
def test_residual_relu_and_streamed_weights(mode):
    """layer2 c2: relu(conv(y) + identity), weights streamed through the ring (+4) and resident."""
    x, w, b, pc = layer(128, 128, 3, 1, 50, seed=7)
    r = rnd(1, N_IMG, 128, 50, 50, seed=9).to(DEV)
    xh, rh = to_hl_dev(x), to_hl_dev(r)
    ref = F.relu(ref_conv(x, w, b, 1) + r.double())
    for g in (3, 7):
        y = dense.conv(xh, pc, relu=True, residual=rh, tune=(mode, g))
        y2 = dense.conv(xh, pc, relu=True, residual=rh, tune=(3, g))
        torch.cuda.synchronize()
        check(hl_f32(y, 128), ref)
        assert torch.equal(y.hi, y2.hi) and torch.equal(y.lo, y2.lo)


@pytest.mark.parametrize("mode", [4, 5])
def test_256_columns_residual_one_launch(mode):
    """layer3 c2 with its residual: both column halves of every tile in one launch, partial output store."""
    x, w, b, pc = layer(256, 256, 3, 1, 25, seed=11)
    r = rnd(1, N_IMG, 256, 25, 25, seed=13).to(DEV)
    xh, rh = to_hl_dev(x), to_hl_dev(r)
    y = dense.conv(xh, pc, relu=True, residual=rh, tune=(mode, 1))
    torch.cuda.synchronize()
    check(hl_f32(y, 256), F.relu(ref_conv(x, w, b, 1) + r.double()))
    out = dense.HL.zeros(1, N_IMG, 25, 25, 256, DEV)
    dense.conv(xh, pc, relu=True, residual=rh, out=out, n_store=192, tune=(mode, 1))   # [192, 256) stay zero
    torch.cuda.synchronize()
    assert torch.equal(out.hi[..., :192], y.hi[..., :192]) and float(out.hi[..., 192:].abs().max()) == 0.0


@pytest.mark.parametrize("mode", [4, 5])
def test_second_destination(mode):
    """bn = 128: columns [64, 128) go to a second tensor with their own activation."""
    x, w, b, pc = layer(64, 128, 3, 1, 50, seed=21)
    xh = to_hl_dev(x)
    o1, o2 = dense.HL.empty(1, N_IMG, 50, 50, 64, DEV), dense.HL.empty(1, N_IMG, 50, 50, 64, DEV)
    dense.conv(xh, pc, out=o1, n_store=64, out2=o2, n_store2=64, relu=False, relu2=True, tune=(mode, 3))
    torch.cuda.synchronize()
    ref = ref_conv(x, w, b, 1)
    check(hl_f32(o1, 64), ref[:, :, :64])
    check(hl_f32(o2, 64), F.relu(ref[:, :, 64:]))


@pytest.mark.parametrize("mode", [4, 5])
@pytest.mark.parametrize("k,stride", [(3, 1), (3, 2), (1, 2)])
def test_tiles_cross_images_and_tail_is_not_written(mode, k, stride):
    """3 images of 10 x 13 = 130 output pixels: the 128-pixel tile [128, 256) (and the pair tile [0, 256)) spans
    images 0 and 1, and the last tile is partial.  The output is a view into a larger sentinel-filled buffer: nothing
    past n_img * Ho * Wo changes."""
    H, W, n_img = 10 * stride, 13 * stride, 3
    x = rnd(1, n_img, 64, H, W, seed=31).to(DEV)
    w = rnd(64, 64, k, k, seed=32, scale=(64 * k * k) ** -0.5).to(DEV)
    b = rnd(64, seed=33).to(DEV)
    pc = dense.pack_conv(w, b, stride=stride)
    n = n_img * 10 * 13 * 64
    sentinel = torch.tensor(-12345.0).to(torch.bfloat16)
    bufs = [torch.full((n + 300 * 64,), float(sentinel), dtype=torch.bfloat16, device=DEV) for _ in range(2)]
    out = dense.HL(bufs[0][:n].view(1, n_img, 10, 13, 64), bufs[1][:n].view(1, n_img, 10, 13, 64), 64)
    dense.conv(to_hl_dev(x), pc, relu=True, out=out, tune=(mode, 1))
    torch.cuda.synchronize()
    check(hl_f32(out, 64), F.relu(ref_conv(x, w, b, stride)))
    for buf in bufs:
        assert bool((buf[n:] == sentinel).all())


def _raises_einval(fn):
    with pytest.raises(RuntimeError, match=r"failed \(-1\)"):
        fn()


@pytest.mark.parametrize("mode", [4, 5])
def test_refused_layers_raise_einval(mode):
    x = to_hl_dev(rnd(1, 3, 64, 20, 20, seed=41).to(DEV))
    w = rnd(64, 64, 3, 3, seed=42, scale=1 / 24).to(DEV)
    b = rnd(64, seed=43).to(DEV)
    pc = dense.pack_conv(w, b)
    t = (mode, 1)
    # temporal taps (dt != 0)
    pc3 = dense.pack_conv(rnd(64, 64, 2, 3, 3, seed=44).to(DEV) / 24, b)
    _raises_einval(lambda: dense.conv(x, pc3, tune=t))
    # a frame window smaller than the whole T axis
    _raises_einval(lambda: dense.conv(x, pc, frames=(1, 2), tune=t))
    # per-image column sums
    cs = torch.empty(3, 64, device=DEV)
    _raises_einval(lambda: dense.conv(x, pc, col_sums=cs, tune=t))
    # fused 1x1 head
    ho = torch.empty(3, 1, 20, 20, device=DEV)
    head = {"w": torch.zeros(1, 64, device=DEV), "b": torch.zeros(1, device=DEV), "outs": [(ho, 0)]}
    _raises_einval(lambda: dense.conv(x, pc, store=False, head=head, tune=t))
    # fp32 outputs (either layout) and per-image bias
    f = torch.empty(3, 64, 20, 20, device=DEV)
    _raises_einval(lambda: dense.conv(x, pc, out_f32=f, n_valid=64, tune=t))
    fn = torch.empty(3, 20, 20, 64, device=DEV)
    _raises_einval(lambda: dense.conv(x, pc, out_f32=fn, n_valid=64, out_f32_nhwc=True, tune=t))
    ib = torch.zeros(3, 64, device=DEV)
    _raises_einval(lambda: dense.conv(x, pc, img_bias=ib, tune=t))
