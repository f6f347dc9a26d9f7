"""tcgen05 (TMA + TMEM, fp16/bf16 operand-split) implicit-GEMM convolution vs fp64 torch CPU convolution."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous().to(_dev())


def _nchw(y):
    return y.permute(0, 3, 1, 2).cpu()


def _cw(w):
    from marconet_b200 import ops
    cout, cin, kh, kw = w.shape
    return ops.ConvWeight(w.permute(2, 3, 1, 0).reshape(kh * kw * cin, cout).contiguous().to(_dev()), kh * kw)


def _ref(x, w, pad):
    return F.conv2d(x.double(), w.double(), padding=pad).float()


TC_CASES = [
    # N, H, W, Cin, Cout, k
    (2, 8, 128, 64, 64, 3),       # TW=128, NT=64
    (1, 64, 64, 128, 128, 3),     # TW=64, TH=2, NT=128
    (3, 32, 32, 64, 256, 3),      # TW=32, TH=4, NT=256
    (5, 4, 4, 64, 64, 3),         # TN=8, ragged last image group
    (16, 8, 8, 128, 512, 3),      # TN=2, two N tiles
    (2, 16, 128, 256, 128, 1),    # 1x1
    (1, 32, 32, 512, 512, 3),     # deep K: 72 k-blocks, many pipeline wraps
    (70, 1, 1, 512, 1024, 1),     # a linear layer: [M,1,1,K]
    (3, 8, 16, 64, 128, 3),       # odd number of pixel tiles: padding CTA inside a 2-CTA cluster
    (1, 64, 1024, 64, 64, 3),     # 512 pixel tiles: several work items per persistent CTA
    (1, 16, 512, 128, 256, 1),    # 1x1 on a wide map, two N tiles
    (4, 8, 8, 512, 512, 3),       # few tiles, deep K: split-K over channel blocks + reduce kernel
    (1, 8, 512, 256, 256, 3),     # ResNet stage at batch 1 (split-K 2)
]
# tensor-core fp32 accumulation truncates (round-toward-zero): the error grows ~linearly with K/16 accumulation steps
TOL = {"f16x3": 4e-5, "bf16x3": 2e-4, "f16x1": 4e-3}


@pytest.mark.parametrize("mode", ["f16x3", "bf16x3", "f16x1"])
@pytest.mark.parametrize("case", TC_CASES)
def test_conv_tc_matches_fp64(case, mode):
    from marconet_b200 import ops
    prec = {"f16x3": ops.PREC_F16X3_TC, "bf16x3": ops.PREC_BF16X3_TC, "f16x1": ops.PREC_F16X1_TC}[mode]
    n, h, w, cin, cout, k = case
    x = _rand(n, cin, h, w, seed=1) * 1.7 + 0.2
    wt = _rand(cout, cin, k, k, seed=2, scale=1.0 / math.sqrt(cin * k * k))
    ref = _ref(x, wt, k // 2)
    y = ops.conv2d(_nhwc(x), _cw(wt), k, k, pad=(k // 2, k // 2), precision=prec)
    torch.cuda.synchronize()
    err = (_nchw(y) - ref).abs().max().item()
    scale = ref.abs().max().item()
    print(f"{mode} {case}: max abs err {err:.3e} (ref max {scale:.2f})")
    assert err <= TOL[mode] * max(1.0, scale)


def test_conv_tc_epilogue_and_slices():
    """demod scale + bias + residual + lrelu*sqrt2 + second (pre-modulated) output + window mask, channel-sliced input."""
    from marconet_b200 import ops
    d = _dev()
    n, h, w, cin, cout = 4, 32, 32, 64, 128
    buf = _rand(n, h, w, 96, seed=3).to(d)
    xin = buf[..., 32:96]
    valid = [32, 20, 7, 32]
    for i, v in enumerate(valid):
        buf[i, :, v:, :] = 0
    x = xin.permute(0, 3, 1, 2).cpu()
    wt = _rand(cout, cin, 3, 3, seed=4, scale=0.05)
    bias, osc, y2s = _rand(cout, seed=5), _rand(n, cout, seed=6).abs() + 0.5, _rand(n, cout, seed=7)
    res = _rand(n, cout, h, w, seed=8)
    y, y2 = ops.conv2d(xin, _cw(wt), 3, 3, pad=(1, 1), bias=bias.to(d), out_scale=osc.to(d), residual=_nhwc(res),
                       act=ops.ACT_LRELU02, gain=2 ** 0.5, out2=True, y2_scale=y2s.to(d),
                       valid_w=torch.tensor(valid, dtype=torch.int32, device=d), precision=ops.PREC_F16X3_TC)
    y, y2 = _nchw(y), _nchw(y2)
    for i, v in enumerate(valid):
        r = _ref(x[i:i + 1, :, :, :v], wt, 1) * osc[i][None, :, None, None] + bias[None, :, None, None] + res[i:i + 1, :, :, :v]
        r = F.leaky_relu(r, 0.2) * 2 ** 0.5
        assert (y[i:i + 1, :, :, :v] - r).abs().max().item() <= 2e-5 * max(1.0, r.abs().max().item())
        assert (y2[i:i + 1, :, :, :v] - r * y2s[i][None, :, None, None]).abs().max().item() <= 4e-5 * max(1.0, r.abs().max().item())
        if v < w:
            assert y[i, :, :, v:].abs().max().item() == 0


@pytest.mark.parametrize("shape", [(3, 32, 32, 128, 128), (1, 16, 256, 64, 64), (5, 16, 16, 256, 128), (2, 8, 8, 64, 64)],
                         ids=["n3_32x32_128to128", "n1_16x256_64to64", "n5_16x16_256to128", "n2_8x8_two_pass_fallback"])
@pytest.mark.parametrize("ragged", [False, True])
def test_conv_tc_fused_groupnorm_swish(ragged, shape):
    """swish(GroupNorm(x)) built inside the conv's operand-split stage == GroupNorm + swish + conv in fp64: 128- and 64-wide tiles,
    several channel blocks, an odd number of samples (padding CTA of the last pair), ragged windows; maps smaller than one 128-pixel
    tile (8x8) take the two-pass form transparently."""
    from marconet_b200 import ops
    d = _dev()
    n, h, w, cin, cout = shape
    x = _rand(n, cin, h, w, seed=20) * 2 + 0.3
    valid = [w, max(1, w // 2 + 1), 5, w - 1, 1][:n] if ragged else None
    if ragged:
        for i, v in enumerate(valid):
            x[i, :, :, v:] = 0
    wt = _rand(cout, cin, 3, 3, seed=21, scale=0.04)
    gamma, beta, bias = _rand(cin, seed=22) * 0.3 + 1, _rand(cin, seed=23) * 0.2, _rand(cout, seed=24)
    vw = torch.tensor(valid, dtype=torch.int32, device=d) if ragged else None
    xn = _nhwc(x)
    mr = ops.groupnorm_stats(xn, valid_w=vw)
    y = ops.conv2d(xn, _cw(wt), 3, 3, pad=(1, 1), bias=bias.to(d), valid_w=vw, gn=(mr, gamma.to(d), beta.to(d)), gn_fuse=True,
                   precision=ops.PREC_F16X3_TC)
    y = _nchw(y)
    for i in range(n):
        v = valid[i] if ragged else w
        xi = x[i:i + 1, :, :, :v].double()
        g = F.group_norm(xi, cin // 32, gamma.double(), beta.double(), eps=1e-6)
        g = g * torch.sigmoid(g)
        ref = F.conv2d(g, wt.double(), bias.double(), padding=1).float()
        err = (y[i:i + 1, :, :, :v] - ref).abs().max().item()
        assert err <= 3e-5 * max(1.0, ref.abs().max().item()), f"sample {i}: {err}"
        if v < w:
            assert y[i, :, :, v:].abs().max().item() == 0


def test_tc_unsupported_shape_is_reported():
    """An explicit tensor-core precision on a 64->64 3x3 geometry the kernel's planner rejects raises, naming the planner's reason."""
    from marconet_b200 import ops
    wt = _rand(64, 64, 3, 3, seed=10)
    for h, w, reason in ((5, 7, "H must be a multiple of 8"), (12, 128, "H must be a multiple of 8"), (2, 256, "halo tile too large")):
        x = _rand(1, 64, h, w, seed=9)
        with pytest.raises(RuntimeError, match="not supported.*" + reason):
            ops.conv2d(_nhwc(x), _cw(wt), 3, 3, pad=(1, 1), precision=ops.PREC_F16X3_TC)
