"""Deterministic synthetic checkpoints and inputs (benchmark / test data generation only: random tensors, no model arithmetic).

The released MARCONet weights are not reachable offline (the reference only
ships checkpoints/download_github.py:1-11), so parity is established on
seeded synthetic state_dicts that carry exactly the reference's keys and
shapes (SURVEY.md section 8b; strict-load into the reference classes is asserted by
oracle/make_golden.py).  Distributions follow the reference constructors
(models/networks.py:182-184,204,240,274-277,311; models/resnet.py:44-47; torch
defaults for Linear/Conv2d/LayerNorm/GroupNorm) with a small perturbation on
tensors that default to all-zeros/all-ones so that every bias/affine path is
exercised.  Spectral-norm u/v vectors are settled with power iterations,
otherwise sigma ~ 0 and the eval forward is NaN (SURVEY.md section 0.6).
"""
import math

import torch
import torch.nn.functional as F


class _Gen:
    def __init__(self, seed):
        self.g = torch.Generator(device="cpu")
        self.g.manual_seed(seed)

    def randn(self, *shape):
        return torch.randn(*shape, generator=self.g, dtype=torch.float32)

    def uniform(self, shape, bound):
        return (torch.rand(*shape, generator=self.g, dtype=torch.float32) * 2 - 1) * bound


# ------------------------------------------------------------------ TSPGAN
_G_RES_CH = {4: 512, 8: 512, 16: 512, 32: 512, 64: 256, 128: 128}


def tspgan_layers():
    """(name, cin, cout, upsample) for the 11 StyledConvs and (name, cin) for the 6 ToRGBs,
    in execution order (models/networks.py:103-132,144-160)."""
    convs = [("conv1", 512, 512, False)]
    rgbs = [("to_rgb1", 512)]
    cin = 512
    for j, res in enumerate((8, 16, 32, 64, 128)):
        cout = _G_RES_CH[res]
        convs.append((f"convs.{2 * j}", cin, cout, True))
        convs.append((f"convs.{2 * j + 1}", cout, cout, False))
        rgbs.append((f"to_rgbs.{j}", cout))
        cin = cout
    return convs, rgbs


def make_tspgan_sd(seed=1234, class_num=6736):
    r = _Gen(seed)
    sd = {}
    g = "TextGenerator."
    for i in range(1, 9):
        sd[f"{g}style_mlp.{i}.weight"] = r.randn(512, 512) / 0.01
        sd[f"{g}style_mlp.{i}.bias"] = r.randn(512) * 5.0  # x lr_mul 0.01 -> 0.05
    sd[g + "input_text.TextEmbeddings"] = r.randn(class_num, 512, 1, 1)
    convs, rgbs = tspgan_layers()

    def add_conv(name, cin, cout):
        sd[f"{g}{name}.bias"] = r.randn(1, cout, 1, 1) * 0.1
        sd[f"{g}{name}.conv.weight"] = r.randn(1, cout, cin, 3, 3)
        sd[f"{g}{name}.conv.modulation.weight"] = r.randn(cin, 512)
        sd[f"{g}{name}.conv.modulation.bias"] = 1.0 + r.randn(cin) * 0.1
        sd[f"{g}{name}.activate.bias"] = r.randn(cout) * 0.1

    def add_rgb(name, cin):
        sd[f"{g}{name}.bias"] = r.randn(1, 3, 1, 1) * 0.1
        sd[f"{g}{name}.conv.weight"] = r.randn(1, 3, cin, 1, 1)
        sd[f"{g}{name}.conv.modulation.weight"] = r.randn(cin, 512)
        sd[f"{g}{name}.conv.modulation.bias"] = 1.0 + r.randn(cin) * 0.1

    # key order mirrors the reference registration order (conv1, to_rgb1, convs.*, to_rgbs.*)
    add_conv(*convs[0][:3])
    add_rgb(*rgbs[0])
    for name, cin, cout, _ in convs[1:]:
        add_conv(name, cin, cout)
    for name, cin in rgbs[1:]:
        add_rgb(name, cin)
    return sd


# ----------------------------------------------------------------- encoder
def make_encoder_sd(seed=2345, num_classes=6736):
    r = _Gen(seed)
    sd = {}

    def conv(name, cout, cin, k):
        sd[name] = r.randn(cout, cin, k, k) * math.sqrt(2.0 / (k * k * cout))

    conv("resnet.conv1.weight", 32, 3, 3)
    inpl = 32
    for li, (planes, nblk) in enumerate(zip((32, 64, 128, 256, 512), (3, 4, 6, 6, 3)), 1):
        for bi in range(nblk):
            p = f"resnet.layer{li}.{bi}."
            conv(p + "conv1.weight", planes, inpl, 1)
            conv(p + "conv2.weight", planes, planes, 3)
            if bi == 0:
                conv(p + "downsample.0.weight", planes, inpl, 1)
            inpl = planes

    def linear(name, out_f, in_f, bias=True):
        b = 1.0 / math.sqrt(in_f)
        sd[name + ".weight"] = r.uniform((out_f, in_f), b)
        if bias:
            sd[name + ".bias"] = r.uniform((out_f,), b)

    def norm(name, n):
        sd[name + ".weight"] = 1.0 + r.randn(n) * 0.1
        sd[name + ".bias"] = r.randn(n) * 0.1

    t = "transformer."
    linear(t + "to_patch_embedding.1", 512, 32768)
    tt = t + "transformer."

    def block(p, mlp):
        norm(p + "0.norm", 512)
        linear(p + "0.to_qkv", 1536, 512, bias=False)
        linear(p + "0.to_out", 512, 512, bias=False)
        norm(p + "1.net.0", 512)
        linear(p + "1.net.1", mlp, 512)
        linear(p + "1.net.3", 512, mlp)

    block(tt + "layers.0.", 1024)
    block(tt + "layers.1.", 1024)
    block(tt + "layers_cls.0.", 1024)
    block(tt + "layers_locs.0.", 512)
    block(tt + "layers_w.0.", 512)
    norm(tt + "linear_seq_maxlen.0", 64)
    linear(tt + "linear_seq_maxlen.1", 16, 64)
    norm(t + "linear_cls.0", 512)
    linear(t + "linear_cls.1", num_classes, 512)
    norm(t + "linear_locs.0", 512)
    linear(t + "linear_locs.1", 256, 512)
    linear(t + "linear_locs.3", 2, 256)
    norm(t + "linear_w.0", 512)
    linear(t + "linear_w.1", 512, 512)
    norm(t + "linear_w_maxlen.0", 64)
    linear(t + "linear_w_maxlen.1", 1, 64)
    return sd


# ---------------------------------------------------------------- TSPSRNet
def tspsr_convs():
    """(key prefix, cin, cout) of every spectral-norm conv, registration order
    (models/networks.py:335-409)."""
    d = 256
    L = [("conv_first_32.0", 3, d // 4), ("conv_first_16.0", d // 4, d // 2),
         ("conv_first_8.0", d // 2, d), ("conv_first_8.2", d, d),
         ("conv_body_16.0", d + d // 2, d), ("conv_body_16.2", d, d),
         ("conv_body_32.0", d + d // 4, d), ("conv_body_32.2", d, d),
         ("conv_up.1", d, d), ("RES:conv_up.3", d, d), ("conv_up.4", d, d),
         ("conv_final.0", d, d // 2), ("conv_final.3", d // 2, d // 4),
         ("RES:conv_final.5", d // 4, d // 4), ("conv_final.6", d // 4, 3),
         ("conv_32_scale.0", d, d), ("conv_32_scale.2", d, d),
         ("conv_32_shift.0", d, d), ("conv_32_shift.2", d, d),
         ("RES:conv_32_fuse.0", 2 * d, d),
         ("conv_32_to256.0", 512, d), ("conv_32_to256.2", d, d),
         ("conv_64_scale.0", d, d), ("conv_64_scale.2", d, d),
         ("conv_64_shift.0", d, d), ("conv_64_shift.2", d, d),
         ("RES:conv_64_fuse.0", 2 * d, d)]
    return L


def make_tspsr_sd(seed=3456, power_iters=30):
    r = _Gen(seed)
    sd = {}

    def sn_conv(p, cin, cout):
        fan_in = cin * 9
        b = 1.0 / math.sqrt(fan_in)
        w = r.uniform((cout, cin, 3, 3), b)
        sd[p + ".bias"] = r.uniform((cout,), b)
        sd[p + ".weight_orig"] = w
        u = F.normalize(r.randn(cout), dim=0, eps=1e-12)
        v = F.normalize(r.randn(fan_in), dim=0, eps=1e-12)
        wm = w.flatten(1)
        threads = torch.get_num_threads()
        torch.set_num_threads(1)        # torch.mv splits its sums by thread count: one thread gives the same u, v on every host
        try:
            for _ in range(power_iters):
                v = F.normalize(torch.mv(wm.t(), u), dim=0, eps=1e-12)
                u = F.normalize(torch.mv(wm, v), dim=0, eps=1e-12)
        finally:
            torch.set_num_threads(threads)
        sd[p + ".weight_u"] = u
        sd[p + ".weight_v"] = v

    def gn(p, n):
        sd[p + ".weight"] = 1.0 + r.randn(n) * 0.1
        sd[p + ".bias"] = r.randn(n) * 0.1

    for name, cin, cout in tspsr_convs():
        if name.startswith("RES:"):
            p = name[4:]
            gn(p + ".norm1", cin)
            sn_conv(p + ".conv1", cin, cout)
            gn(p + ".norm2", cout)
            sn_conv(p + ".conv2", cout, cout)
            if cin != cout:
                b = 1.0 / math.sqrt(cin)
                sd[p + ".conv_out.weight"] = r.uniform((cout, cin, 1, 1), b)
                sd[p + ".conv_out.bias"] = r.uniform((cout,), b)
        else:
            sn_conv(name, cin, cout)
    return sd


_CACHE = {}


def make_checkpoints(seed=0):
    """{'tspgan','encoder','sr'} -> reference-format state_dicts (fp32, CPU). Cached per seed."""
    if seed not in _CACHE:
        _CACHE[seed] = dict(tspgan=make_tspgan_sd(1234 + seed), encoder=make_encoder_sd(2345 + seed),
                            sr=make_tspsr_sd(3456 + seed))
    return _CACHE[seed]


# ------------------------------------------------------------------ inputs
def make_lq(batch=1, seed=0):
    """Synthetic LR lines, SURVEY.md section 8d config 2/4: clamp(randn,-1,1), one seed per line."""
    lines = []
    for b in range(batch):
        g = torch.Generator(device="cpu")
        g.manual_seed(seed + b)
        lines.append(torch.randn(1, 3, 32, 512, generator=g).clamp_(-1, 1))
    return torch.cat(lines, 0)


def make_labels(n, seed=0, class_num=6735):
    g = torch.Generator(device="cpu")
    g.manual_seed(1000 + seed)
    return torch.randint(0, class_num, (n, 1), generator=g, dtype=torch.int64)


def make_styles(n, seed=0):
    g = torch.Generator(device="cpu")
    g.manual_seed(2000 + seed)
    return torch.randn(n, 512, generator=g)


def make_locs(batch, n_chars, ragged=False, seed=0):
    """locs[b, 2i] = centre/512, locs[b, 2i+1] = half-width/512 (test_sr.py:121-135).
    Regular grid (config 2) or a jittered/edge-hugging layout that produces clipped and
    overlapping windows."""
    locs = torch.zeros(batch, 2 * n_chars, dtype=torch.float32)
    g = torch.Generator(device="cpu")
    g.manual_seed(3000 + seed)
    for b in range(batch):
        for i in range(n_chars):
            c = (i + 0.5) * 32.0 / 512.0
            if ragged:
                c = (i + 0.5) * (512.0 / n_chars) / 512.0 * 0.97 + 0.004 + float(torch.rand(1, generator=g)) * 0.02
                if i == 0:
                    c = 5.3 / 512.0
                if i == n_chars - 1:
                    c = 506.7 / 512.0
            locs[b, 2 * i] = c
            locs[b, 2 * i + 1] = 14.0 / 512.0
    return locs
