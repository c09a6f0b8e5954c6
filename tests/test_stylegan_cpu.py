"""StyleGAN (v1) on the host: the module tree and random init against the reference (fixture written by
oracle/gen_golden_sg1.py), and the bias identity that lets G_mapping run on the packed StyleGAN2 mapping kernels."""
import math

import numpy as np
import pytest
import torch


@pytest.mark.parametrize("outclass,res", [("ffhq", 1024), ("bedrooms", 256)])
def test_module_tree_and_random_init_match_reference(golden, outclass, res):
    from ganspace_b200.models.stylegan import StyleGAN_G
    g = golden("sg1_mapping_known_answers.npz")
    torch.manual_seed(1234)
    G = StyleGAN_G(res)
    assert [n for n, _ in G.named_modules()] == list(g[f"{outclass}_module_names"])
    assert [n for n, _ in G.named_buffers()] == list(g[f"{outclass}_buffer_names"])
    params = list(G.named_parameters())
    assert [n for n, _ in params] == list(g[f"{outclass}_param_names"])
    # bit-for-bit init: float64 sums of the same float32 values agree to the last bits of the double sum
    sums = np.array([p.detach().double().sum().item() for _, p in params])
    abs_sums = np.array([p.detach().double().abs().sum().item() for _, p in params])
    assert np.allclose(sums, g[f"{outclass}_param_sums"], rtol=1e-12, atol=1e-9)
    assert np.allclose(abs_sums, g[f"{outclass}_param_abs_sums"], rtol=1e-12, atol=1e-9)


def _reference_layer(x, W, b):
    """models/stylegan/model.py:26-49 + nn.LeakyReLU(0.2): lrelu(x (W w_mul)^T + b_mul b), use_wscale, lrmul 0.01."""
    w_mul = math.sqrt(2) * 512 ** -0.5 * 0.01
    y = x @ (W * w_mul).T + 0.01 * b
    return np.where(y >= 0, y, 0.2 * y)


def _packed_layer(x, W, b_packed):
    """The packed mapping kernels' layer (stylegan2-pytorch EqualLinear + fused_lrelu): sqrt2 lrelu(x (W 0.01/sqrt512)^T + 0.01 b)."""
    y = x @ (W * (0.01 / math.sqrt(512))).T + 0.01 * b_packed
    return math.sqrt(2) * np.where(y >= 0, y, 0.2 * y)


def test_g_mapping_bias_identity():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((64, 512))
    W = rng.standard_normal((512, 512)) * 100.0
    b = rng.standard_normal(512) * 30.0          # non-zero, large enough to flip signs of the pre-activation
    ref = _reference_layer(x, W, b)
    assert np.abs(ref - _packed_layer(x, W, b / math.sqrt(2))).max() < 1e-12 * np.abs(ref).max()
    assert np.abs(ref - _packed_layer(x, W, b)).max() > 1e-3 * np.abs(ref).max()     # without the rescale they differ


def test_oracle_mapping_with_rescaled_bias_matches_reference(golden, oracle):
    """The reference's G_mapping outputs (fixture (a)) from the StyleGAN2-form restatement with b' = b/sqrt2."""
    from ganspace_b200.models.stylegan import StyleGAN_G
    g = golden("sg1_mapping_known_answers.npz")
    torch.manual_seed(1234)
    G = StyleGAN_G(256)
    lins = G.g_mapping.dense_layers()
    ws = [l.weight.detach().numpy() for l in lins]
    bs = [(l.bias.detach() / math.sqrt(2.0)).numpy() for l in lins]
    assert np.array_equal(oracle.standard_normal_f32(77, 4 * 512).reshape(4, 512), g["z"])
    w = oracle.mapping_forward_np(g["z"], ws, bs, lr_mul=0.01)
    assert np.abs(w - g["w"]).max() < 2e-5 * max(1.0, np.abs(g["w"]).max())
    assert np.array_equal(g["dense0_act_last"], g["w"])


def _perturbed_generator(ka):
    """Our module tree on the host with the fixture's random init and perturbation (generator order = parameter order)."""
    from ganspace_b200.models.stylegan import StyleGAN_G
    torch.manual_seed(1234)
    G = StyleGAN_G(1024)
    names = set(str(x) for x in ka["perturbed"])
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for k, p in G.named_parameters():
            if k in names:
                p.copy_(float(ka["perturb_scale"]) * torch.randn(p.shape, generator=g))
    return G


def test_tap_form_oracle_vs_reference_activations(golden, oracle):
    """The float64 per-tap restatement of the synthesis layers (both up-sampling variants) against the reference's own
    activations (fixture (b)), up to the first fused transposed-conv block; one latent."""
    from oracle import sg1_oracle as so
    ka = golden("sg1_synthesis_known_answers.npz")
    G = _perturbed_generator(ka)
    lins = G.g_mapping.dense_layers()
    w = oracle.mapping_forward_np(ka["z"][:1], [l.weight.detach().numpy() for l in lins],
                                  [(l.bias.detach() / math.sqrt(2.0)).numpy() for l in lins], lr_mul=0.01)
    sd = {k: v.numpy() for k, v in G.state_dict().items()}
    plan = so.layer_plan(1024)
    layers, rgb = so.params_from_state(sd, 1024)
    noises = {}
    for r in sorted({p[4] for p in plan}):
        torch.manual_seed(0)
        noises[r] = torch.randn(1, 1, r, r)[0, 0].double().numpy()      # StyleGAN.set_noise_seed(0), wrappers.py:420-436
    wl = np.repeat(w.astype(np.float64)[:, None, :], len(layers), axis=1)
    stops = {"blocks_4x4": (1, "epi"), "blocks_8x8_conv0_up": (2, "conv"), "blocks_16x16_epi1": (4, "epi"),
             "blocks_64x64": (9, "epi"), "blocks_32x32_epi2_style_mod_lin": (7, "style"), "blocks_128x128_conv0_up": (10, "conv")}
    for key, (j, what) in stops.items():
        out = so.synthesis(wl, layers[:j + 1], rgb, noises, stop=(j, what))
        if out.ndim == 4:
            out = np.transpose(out, (0, 3, 1, 2))
            step = max(1, out.shape[-1] // 16)
            out = out[:, ::max(1, out.shape[1] // 16), ::step, ::step]
        ref = ka[f"act_{key}_sub"][:1]
        assert out.shape == ref.shape, key
        assert np.abs(out - ref).max() < 2e-5 * np.abs(ref).max(), (key, np.abs(out - ref).max() / np.abs(ref).max())
