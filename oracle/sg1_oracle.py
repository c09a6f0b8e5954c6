"""ORACLE -- StyleGAN (v1) synthesis restated on the host in the per-tap NHWC form the CUDA kernels use (csrc/synthesis_sg1.cu).

Reference form: /root/reference/models/stylegan/model.py:51-104 (MyConv2d, incl. the fused 4x4 transposed conv of :82-91),
:106-122 (NoiseLayer), :124-136 (StyleMod), :145-169 (BlurLayer), :171-188 (Upscale2d), :230-303 (LayerEpilogue, InputBlock,
GSynthesisBlock), :305-363 (G_synthesis).  Tap form, per conv layer with input x [n, H, W, ci]:
    Y[n, i, j, tap, co] = sum_ci x[n, i, j, ci] Wt[tap, co, ci]                       (one dense product: the tap GEMM)
    same (3x3, pad 1):        out[y, x]  = sum_{ky,kx} Y[y + ky - 1, x + kx - 1, (ky, kx)]
    nearest x2 then 3x3:      out[y, x]  = sum_{ky,kx} Y[(y + ky - 1) // 2, (x + kx - 1) // 2, (ky, kx)],  0 <= y + ky - 1 < 2H
    fused transposed (4x4 taps, stride 2, pad 1, w4 = the reference's 4-way summed kernel):
                              out[u, v]  = sum_{ky,kx: u + 1 - ky, v + 1 - kx even} Y[(u + 1 - ky) / 2, (v + 1 - kx) / 2, (ky, kx)]
then (up-sampling layers) the [1,2,1] x [1,2,1] / 16 blur with pad 1, + bias  (= the conv module's output), + noise_w[c] noise[y, x],
lrelu 0.2, instance norm (eps 1e-5, biased variance), StyleMod x (s0 + 1) + s1 with s = lin(w).
Everything is float64 here: it is the accuracy yardstick, and it is pinned to the reference's float32 CPU form in
tests/test_stylegan_cpu.py.
"""
import math

import numpy as np

BLUR = np.outer([1.0, 2.0, 1.0], [1.0, 2.0, 1.0]) / 16.0


def layer_plan(resolution):
    """[(block name, kind, cin, cout, res_out)] of the 2 * log2(res) - 2 layers; kind: 'const' (4x4 epi1), 'same', 'nearest',
    'fused'.  Layer j reads latent j."""
    nf = lambda stage: min(int(8192 / (2.0 ** stage)), 512)
    plan = []
    for r in range(2, int(np.log2(resolution)) + 1):
        name, c, res = f"{2 ** r}x{2 ** r}", nf(r - 1), 2 ** r
        if r == 2:
            plan += [(name, "const", c, c, 4), (name, "same", c, c, 4)]
        else:
            plan += [(name, "fused" if res >= 128 else "nearest", nf(r - 2), c, res), (name, "same", c, c, res)]
    return plan


def fused_kernel(W):
    """model.py:85-89: w = W^T-permuted [ci, co, 3, 3] (already times w_mul), padded by 1, the four shifted sums -> [ci, co, 4, 4]."""
    w = np.transpose(W, (1, 0, 2, 3))
    w = np.pad(w, ((0, 0), (0, 0), (1, 1), (1, 1)))
    return w[:, :, 1:, 1:] + w[:, :, :-1, 1:] + w[:, :, 1:, :-1] + w[:, :, :-1, :-1]


def conv_taps(x, W, kind):
    """Conv of x [n, H, W, ci] (NHWC, float64) in the tap form; W [co, ci, 3, 3] times w_mul.  No bias."""
    n, H, Wd, ci = x.shape
    co = W.shape[0]
    if kind == "fused":
        w4 = fused_kernel(W)                                          # [ci, co, 4, 4]
        Wt = np.transpose(w4, (2, 3, 1, 0)).reshape(16, co, ci)      # tap = ky * 4 + kx
        k = 4
    else:
        Wt = np.transpose(W, (2, 3, 0, 1)).reshape(9, co, ci)
        k = 3
    Y = np.einsum("nijc,toc->nijto", x, Wt)                          # the tap GEMM
    R = H if kind == "same" else 2 * H
    out = np.zeros((n, R, R, co))
    for ky in range(k):
        for kx in range(k):
            t = ky * k + kx
            if kind == "same":
                ys = np.arange(R) + ky - 1
                xs = np.arange(R) + kx - 1
                yi, xi = ys, xs
            elif kind == "nearest":
                ys = np.arange(R) + ky - 1
                xs = np.arange(R) + kx - 1
                yi, xi = np.floor_divide(ys, 2), np.floor_divide(xs, 2)
            else:
                ys = np.arange(R) + 1 - ky
                xs = np.arange(R) + 1 - kx
                yi, xi = ys // 2, xs // 2
            vy = (ys >= 0) & (ys < (R if kind != "fused" else 2 * H)) & (yi < H)
            vx = (xs >= 0) & (xs < (R if kind != "fused" else 2 * H)) & (xi < Wd)
            if kind == "fused":
                vy &= (ys % 2 == 0)
                vx &= (xs % 2 == 0)
            oy, ox = np.nonzero(vy)[0], np.nonzero(vx)[0]
            out[:, oy[:, None], ox[None, :], :] += Y[:, yi[oy][:, None], xi[ox][None, :], t, :]
    return out


def blur(x):
    n, R, _, c = x.shape
    p = np.pad(x, ((0, 0), (1, 1), (1, 1), (0, 0)))
    out = np.zeros_like(x)
    for i in range(3):
        for j in range(3):
            out += BLUR[i, j] * p[:, i:i + R, j:j + R, :]
    return out


def params_from_state(sd, resolution):
    """Per-layer float64 parameters from a StyleGAN_G state dict (numpy arrays keyed like the reference's)."""
    g = lambda k: np.asarray(sd[k], np.float64)
    layers = []
    for j, (name, kind, ci, co, res) in enumerate(layer_plan(resolution)):
        pre = f"g_synthesis.blocks.{name}"
        epi = f"{pre}.epi{1 + j % 2}"
        L = dict(kind=kind, name=name, cin=ci, cout=co, res=res,
                 noise_w=g(f"{epi}.top_epi.noise.weight"),
                 style_w=g(f"{epi}.style_mod.lin.weight") / math.sqrt(512), style_b=g(f"{epi}.style_mod.lin.bias"))
        if kind == "const":
            L["const"] = np.transpose(g(f"{pre}.const")[0], (1, 2, 0))         # [4, 4, c]
            L["bias"] = g(f"{pre}.bias")
        else:
            conv = f"{pre}.conv" if name == "4x4" else (f"{pre}.conv0_up" if j % 2 == 0 else f"{pre}.conv1")
            L["conv"] = conv
            L["W"] = g(f"{conv}.weight") * (math.sqrt(2) / math.sqrt(ci * 9))
            L["bias"] = g(f"{conv}.bias")
        layers.append(L)
    c = layers[-1]["cout"]
    rgb = dict(W=g("g_synthesis.torgb.weight")[:, :, 0, 0] / math.sqrt(c), b=g("g_synthesis.torgb.bias"))
    return layers, rgb


def synthesis(w_layers, layers, rgb, noises, stop=None):
    """w_layers [n, n_layers, 512] (float64); noises[res] = [res, res] map.  ``stop`` = (layer index, what) with what in
    'conv' (conv module output), 'epi' (epilogue output), 'style' (StyleMod style vector); None -> the torgb image NCHW."""
    n = w_layers.shape[0]
    x = None
    for j, L in enumerate(layers):
        if L["kind"] == "const":
            c = np.broadcast_to(L["const"] + L["bias"], (n,) + L["const"].shape).copy()
        else:
            c = conv_taps(x, L["W"], L["kind"])
            if L["kind"] != "same":
                c = blur(c)
            c = c + L["bias"]
        if stop == (j, "conv"):
            return c
        a = c + L["noise_w"] * noises[L["res"]][None, :, :, None]
        a = np.where(a >= 0, a, 0.2 * a)
        mean = a.mean(axis=(1, 2), keepdims=True)
        var = ((a - mean) ** 2).mean(axis=(1, 2), keepdims=True)
        a = (a - mean) / np.sqrt(var + 1e-5)
        s = w_layers[:, j] @ L["style_w"].T + L["style_b"]
        if stop == (j, "style"):
            return s
        co = L["cout"]
        x = a * (s[:, None, None, :co] + 1) + s[:, None, None, co:]
        if stop == (j, "epi"):
            return x
    img = x @ rgb["W"].T + rgb["b"]
    return np.transpose(img, (0, 3, 1, 2))
