"""GPU (B200): the backward building blocks, each through the C ABI, against torch autograd on the
same bf16-rounded operands (fp32 accumulation on both sides)."""
import pytest
import torch
import torch.nn.functional as F

from helpers import C_TC, abs_conv, assert_bf16_elementwise, ref_conv, rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from xmm_superres_denoise_b200 import _lib

    _lib.check(_lib.load().xmm_check_device())
    return torch.device("cuda:0")


def _ref_wgrad(x_nhwc, dy_nhwc):
    """dW[o][i][3][3] of conv2d(x, W, padding=1) given dL/dy, via autograd (fp32)."""
    x = x_nhwc.float().permute(0, 3, 1, 2).contiguous()
    dy = dy_nhwc.float().permute(0, 3, 1, 2).contiguous()
    w = torch.zeros(dy.shape[1], x.shape[1], 3, 3, requires_grad=True)
    F.conv2d(x, w, padding=1).backward(dy)
    return w.grad


@pytest.mark.parametrize("stacked,h,w", [(0, 40, 24), (1, 40, 24), (1, 37, 29)])
def test_wgrad_dense_block_roles(dev, stacked, h, w):
    """X = 160-channel activation buffer, dY = 160-channel gradient buffer (slot k-1 = dY_k):
    3 main roles (x0..x3 against all dY) + tail role (x4 against dY_5), 16 destinations.  The tail either as nine
    N=32 taps or as a "stacked" role (operands swapped, three dx taps per MMA as overlapping swizzle atoms)."""
    from xmm_superres_denoise_b200 import ops

    g = torch.Generator().manual_seed(0)
    b, f = 2, 32  # (37 x 29: ragged against the 8 x 8 pixel tiles -- out-of-image rows / columns are TMA zero fill)
    x = torch.randn(b, h, w, 5 * f, generator=g).to(torch.bfloat16)
    dy = (torch.randn(b, h, w, 5 * f, generator=g) * 0.1).to(torch.bfloat16)
    roles = [(3 * d, 3, 0, 2, 0, 160) for d in range(3)]
    roles.append((0, 3, 128, 1, 96, 96, 1) if stacked else (0, 9, 128, 1, 128, 32))
    dws = [torch.full((f, k * f, 3, 3), 7.0, device=dev) for k in range(1, 6)]
    dsts = []
    for k in range(1, 6):
        scale = 0.2 if k == 5 else 1.0
        for d in range(3):
            dsts.append((dws[k - 1], f, k * f, 0, min(k * f, 128), d, 0, (k - 1) * f, scale, 0, 0))
    dsts.append((dws[4], f, 5 * f, 128, 160, 3, 32 if stacked else 0, 0, 0.2, 0, 0))
    ops.conv3x3_wgrad(x.to(dev), dy.to(dev), roles, dsts)
    torch.cuda.synchronize()
    for k in range(1, 6):
        want = _ref_wgrad(x[..., :k * f], dy[..., (k - 1) * f:k * f]) * (0.2 if k == 5 else 1.0)
        assert rel_l2(dws[k - 1].cpu(), want) < 2e-3, k


@pytest.mark.parametrize("stacked", [0, 1])
@pytest.mark.parametrize("n,perm", [(32, 0), (128, 1)])
def test_wgrad_single_conv(dev, n, perm, stacked):
    """F -> n convolution whose input tensor has only F=32 channels (TMA zero-fills channels 32..63)."""
    from xmm_superres_denoise_b200 import ops

    g = torch.Generator().manual_seed(n)
    b, h, w, f = 1, 32, 40, 32
    x = torch.randn(b, h, w, f, generator=g).to(torch.bfloat16)
    dy = (torch.randn(b, h, w, n, generator=g) * 0.1).to(torch.bfloat16)
    dw = torch.zeros(n, f, 3, 3, device=dev)
    dw += 1.0
    if stacked:  # operands swapped: lanes = the n dY channels (1 or 2 boxes), columns = 3 dx taps x 32 X channels
        roles = [(0, 3, 0, 1 if n <= 64 else 2, 0, 96, 1)]
        dsts = [(dw, n, f, 0, f, 0, 0, 0, 1.0, 1, perm)]
    elif n == 32:
        roles = [(0, 9, 0, 1, 0, 32)]
        dsts = [(dw, n, f, 0, f, 0, 0, 0, 1.0, 1, perm)]
    else:
        roles = [(3 * d, 3, 0, 1, 0, 128) for d in range(3)]
        dsts = [(dw, n, f, 0, f, d, 0, 0, 1.0, 1, perm) for d in range(3)]
    ops.conv3x3_wgrad(x.to(dev), dy.to(dev), roles, dsts)
    want = _ref_wgrad(x, dy)
    if perm:  # packed column g*32+c holds PixelShuffle channel 4c+g
        idx = torch.tensor([4 * (j % 32) + j // 32 for j in range(n)])
        full = torch.zeros_like(want)
        full[idx] = want
        want = full
    assert rel_l2(dw.cpu() - 1.0, want) < 2e-3


def test_colsum(dev):
    from xmm_superres_denoise_b200 import ops

    x = torch.randn(3, 17, 23, 160).to(torch.bfloat16)
    out = torch.full((32,), 5.0, device=dev)
    ops.colsum(x.to(dev), 64, 32, out, scale=0.2)
    want = x[..., 64:96].float().sum(dim=(0, 1, 2)) * 0.2
    assert rel_l2(out.cpu(), want) < 1e-4
    ops.colsum(x.to(dev), 64, 32, out, scale=1.0, accumulate=True)
    assert rel_l2(out.cpu(), want * 6.0) < 1e-4


def test_conv_last_backward_pieces(dev):
    """conv_last data gradient = conv_first stencil with transposed/flipped weights, gated by the
    clamp and masked by LeakyReLU'; weight/bias gradient = edge_wgrad."""
    from xmm_superres_denoise_b200 import ops

    g = torch.Generator().manual_seed(1)
    b, h, w, f = 2, 21, 19, 32
    u = torch.randn(b, h, w, f, generator=g).to(torch.bfloat16)       # conv_last input (post-LeakyReLU values)
    wl = (torch.randn(1, f, 3, 3, generator=g) * 0.1).requires_grad_(True)
    bl = torch.zeros(1, requires_grad=True)
    pre_act = u.float().permute(0, 3, 1, 2).clone().requires_grad_(True)
    pre = F.conv2d(pre_act, wl, bl, padding=1) * 3.0
    out = pre.clamp(0, 1)
    gout = torch.randn(b, 1, h, w, generator=g)
    out.backward(gout)
    # data gradient w.r.t. the activation feeding conv_last, times LeakyReLU'(0.2) of that activation
    want_du = pre_act.grad / 3.0 * torch.where(pre_act.detach() > 0, 1.0, 0.2)
    wt = wl.detach().flip(2, 3).permute(1, 0, 2, 3).contiguous().to(dev)
    du = torch.empty(b, h, w, f, dtype=torch.bfloat16, device=dev)
    ops.conv_first(gout.to(dev), wt, None, du, 0, gate=pre.detach().to(dev), mask=u.to(dev), mask_coff=0, mask_slope=0.2)
    assert rel_l2(du.float().permute(0, 3, 1, 2).cpu(), want_du) < 5e-3
    r = torch.zeros(1, f, 9, device=dev)
    ssum = torch.zeros(1, device=dev)
    ops.edge_wgrad(gout.to(dev), u.to(dev), 0, f, r, ssum=ssum, gate=pre.detach().to(dev))
    assert rel_l2(r.reshape(1, f, 3, 3).cpu(), wl.grad / 3.0) < 1e-4
    assert rel_l2(ssum.cpu(), bl.grad / 3.0) < 1e-4


def test_conv_first_weight_gradient_via_edge_wgrad(dev):
    from xmm_superres_denoise_b200 import ops

    g = torch.Generator().manual_seed(2)
    b, h, w, f = 2, 18, 26, 32
    x = torch.rand(b, 1, h, w, generator=g)
    x[x < 0.5] = 0
    dfa = (torch.randn(b, h, w, f, generator=g) * 0.1).to(torch.bfloat16)
    dfb = (torch.randn(b, h, w, f, generator=g) * 0.1).to(torch.bfloat16)
    wf = torch.zeros(f, 1, 3, 3, requires_grad=True)
    F.conv2d(x, wf, padding=1).backward((dfa.float() + dfb.float()).permute(0, 3, 1, 2))
    r = torch.zeros(1, f, 9, device=dev)
    ops.edge_wgrad(x.to(dev), dfa.to(dev), 0, f, r, v2=dfb.to(dev), v2_coff=0)
    got = r.cpu().reshape(f, 9).flip(1).reshape(f, 1, 3, 3)  # dW_first[f][0][8 - tap] = R[0][f][tap]
    assert rel_l2(got, wf.grad) < 1e-4


def test_conv3x3_inverse_pixel_shuffle_store(dev):
    from xmm_superres_denoise_b200 import ops
    from xmm_superres_denoise_b200.engine import WeightArena, _Blob, _Segment

    g = torch.Generator().manual_seed(3)
    b, h, w, f = 1, 32, 16, 32
    x = torch.randn(b, h, w, f, generator=g).to(torch.bfloat16)
    wgt = (torch.randn(f, f, 3, 3, generator=g) * 0.05).to(dev)
    arena = WeightArena()
    arena.add(_Blob("c", f, 32, 1, [_Segment(wgt, f, 0, 0, 0, 0, f, 1.0)], None))
    arena.ensure(dev)
    out = torch.zeros(b, h // 2, w // 2, 4 * f, dtype=torch.bfloat16, device=dev)
    ops.conv3x3(x.to(dev), 0, f, arena.ptr("c"), 32, f, out, 0, pixel_shuffle=2)
    torch.cuda.synchronize()
    xin, wq = x.permute(0, 3, 1, 2), wgt.cpu().to(torch.bfloat16)

    def unshuffle(t):  # [b,f,h,w] -> [b,4f,h/2,w/2], channel (2*(y&1) + (x&1)) * f + c
        return t.reshape(b, f, h // 2, 2, w // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(b, 4 * f, h // 2, w // 2)

    r = assert_bf16_elementwise(out.cpu().permute(0, 3, 1, 2), unshuffle(ref_conv(xin, wq)), unshuffle(abs_conv(xin, wq)),
                                C_TC, what="inverse pixel-shuffle store")
    print(f"inverse pixel-shuffle store: max |err|/bound = {r:.3f}")
