"""StyleGAN (v1) on the B200: the wrapper, g_mapping on the packed mapping kernels, hooks on g_mapping and its children, the
fused synthesis chain (activations, images, hooks) and get_or_compute on g_mapping (Z and W space) and on a synthesis block,
against the unmodified reference's fixtures (oracle/gen_golden_sg1.py)."""
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_TOL = 0.999        # sign-normalised cosine >= 0.999 per component
RATIO_TOL = 1e-3       # explained-variance ratios within 1e-3
AUX_TOL = 1e-4         # means / stdevs: fp32-grade (tcgen05 mapping path, see test_e2e_gpu.py)
MAP_TOL = 1e-4         # mapping outputs, relative to their max
ACT_TOL = 5e-4         # synthesis activations after up to 18 layers, relative to their max (as the StyleGAN2 render tests)
IMG_TOL = 1e-3         # images, relative to their max


@pytest.fixture(scope="module")
def model():
    from ganspace_b200.models import StyleGAN
    return StyleGAN(torch.device("cuda:0"), "ffhq", random_init=1234)


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_get_model_constructs_stylegan(model):
    from ganspace_b200.models import get_model
    assert get_model("StyleGAN", "ffhq", torch.device("cuda:0"), model=model) is model
    assert model.get_max_latents() == 18 and model.latent_space_name() == "Z" and model.name == "StyleGAN-ffhq"
    with pytest.raises(RuntimeError, match="cannot change output class"):
        model.set_output_class("cars")
    with pytest.raises(RuntimeError, match="outside the B200 hot path"):
        get_model("ProGAN", "churchoutdoor", torch.device("cuda:0"))


def test_sample_latent_and_mapping_vs_reference(model, golden):
    g = golden("sg1_mapping_known_answers.npz")
    model.use_z()
    z = model.sample_latent(4, seed=77)
    assert np.array_equal(z.cpu().numpy(), g["z"])
    np.random.seed(5)
    assert np.array_equal(model.sample_latent(2).cpu().numpy(), g["z_global_seed5"])
    w = model.model.g_mapping(z)
    assert _rel(w.cpu().numpy(), g["w"]) < MAP_TOL
    model.use_w()
    try:
        assert _rel(model.sample_latent(4, seed=77).cpu().numpy(), g["w_sample_seed77"]) < MAP_TOL
    finally:
        model.use_z()
    model.check_numerics()


def test_g_mapping_child_hooks_retain_and_edit(model, golden):
    from ganspace_b200.netdissect.nethook import InstrumentedModel
    g = golden("sg1_mapping_known_answers.npz")
    model.use_z()
    z = torch.from_numpy(g["z"]).cuda()
    with InstrumentedModel(model) as inst:
        inst.retain_layers(["g_mapping", "g_mapping.dense3", "g_mapping.dense0_act"])
        model.partial_forward(z, "g_mapping")
        assert _rel(inst.retained_layer("g_mapping.dense3").cpu().numpy(), g["dense3"]) < MAP_TOL
        assert _rel(inst.retained_layer("g_mapping.dense0_act").cpu().numpy(), g["w"]) < MAP_TOL
        w_layers = inst.retained_layer("g_mapping").clone()
        assert _rel(w_layers.cpu().numpy(), g["w"]) < MAP_TOL
        # an edit on a child propagates through the remaining layers; an edit on g_mapping is what the caller receives
        inst.edit_layer("g_mapping.dense7", offset=torch.full((512,), 3.0, device="cuda"))
        model.partial_forward(z, "g_mapping")
        assert (inst.retained_layer("g_mapping") - w_layers).abs().min() > 0.5
    with InstrumentedModel(model) as inst:
        inst.edit_layer("g_mapping", offset=torch.ones(512, device="cuda"))
        out = model.model.g_mapping(z)
        assert torch.allclose(out, w_layers + 1, rtol=0, atol=MAP_TOL * float(w_layers.abs().max()))


def test_set_noise_seed_matches_reference_draws(model):
    from ganspace_b200.models import stylegan
    model.set_noise_seed(4)
    for name, m in model.model.named_modules(remove_duplicate=False):
        if isinstance(m, stylegan.NoiseLayer):
            res = int(name.split(".")[2].split("x")[0])
            torch.manual_seed(4)
            assert torch.equal(m.noise.cpu(), torch.randn(1, 1, res, res))
    model.set_noise_seed(0)


@pytest.mark.parametrize("use_w", [False, True], ids=["z", "w"])
def test_get_or_compute_g_mapping_vs_reference(model, golden, oracle, use_w):
    from ganspace_b200.config import Config
    from ganspace_b200.decomposition import get_or_compute
    from ganspace_b200.models import get_instrumented_model
    g = golden(f"sg1_ffhq_g_mapping_{'w' if use_w else 'z'}_n10000_b1000_c32.npz")
    cfg = Config(output_class="ffhq", n=10_000, batch_size=1_000, components=32, use_w=use_w)
    assert (cfg.model, cfg.layer, cfg.estimator) == ("StyleGAN", "g_mapping", "ipca")
    inst = get_instrumented_model(cfg, torch.device("cuda:0"), model=model)
    try:
        with tempfile.TemporaryDirectory() as tmp:
            path = get_or_compute(cfg, inst, submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp), force_recompute=True)
            with np.load(path, allow_pickle=False) as data:
                out = {k: data[k] for k in data.files}
    finally:
        inst.close()
        model.use_z()
    assert path.name == str(g["dump_name"])
    for k in ("act_comp", "act_mean", "act_stdev", "lat_comp", "lat_mean", "lat_stdev", "var_ratio", "random_stdevs"):
        assert out[k].shape == g[k].shape and out[k].dtype == np.float32, k
    cmp = oracle.compare_npz(out, g)
    assert cmp["min_signed_cos"] >= COS_TOL and cmp["min_lat_signed_cos"] >= COS_TOL, cmp
    assert cmp["max_abs_dvar_ratio"] <= RATIO_TOL, cmp
    for k in ("act_mean_rel", "act_stdev_rel", "lat_mean_rel", "lat_stdev_rel", "random_stdevs_rel"):
        assert cmp[k] < AUX_TOL, (k, cmp)
    model.check_numerics()


# ---- synthesis --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ka(golden):
    return golden("sg1_synthesis_known_answers.npz")


@pytest.fixture(scope="module")
def synth(ka):
    """The fixture's model: random init 1234 with the zero-initialised synthesis parameters perturbed in the generator's order."""
    from ganspace_b200.models import StyleGAN
    m = StyleGAN(torch.device("cuda:0"), "ffhq", random_init=1234)
    names = set(str(x) for x in ka["perturbed"])
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for k, p in m.model.named_parameters():
            if k in names:
                p.copy_(float(ka["perturb_scale"]) * torch.randn(p.shape, generator=g))
    m.set_noise_seed(0)
    m.use_z()
    return m


def _sub(act, grid):
    """The fixture's subsample: every (C // 16)-th channel on a grid x grid raster."""
    if act.ndim == 4:
        step = max(1, act.shape[-1] // grid)
        return act[:, ::max(1, act.shape[1] // 16), ::step, ::step]
    return act


def _check_known(ka, key, act, tol, grid=16):
    act = act.detach().cpu().numpy() if torch.is_tensor(act) else act
    assert tuple(act.shape) == tuple(ka[f"shape_{key}"]), key
    assert _rel(_sub(act, grid), ka[f"act_{key}_sub"]) < tol, (key, _rel(_sub(act, grid), ka[f"act_{key}_sub"]))
    sums = np.array([act.astype(np.float64).sum(), (act.astype(np.float64) ** 2).sum()])
    assert abs(sums[1] - ka[f"sum_{key}"][1]) < tol * ka[f"sum_{key}"][1], (key, sums, ka[f"sum_{key}"])


def test_partial_forward_activations_vs_reference(synth, ka):
    from ganspace_b200.netdissect.nethook import InstrumentedModel
    z = torch.from_numpy(ka["z"]).cuda()
    for layer in [str(x) for x in ka["layers"]]:
        if layer == "g_synthesis.torgb":
            continue
        with InstrumentedModel(synth) as inst:
            inst.retain_layer(layer)
            synth.partial_forward(z, layer)
            _check_known(ka, layer.replace("g_synthesis.", "").replace(".", "_"), inst.retained_layer(layer), ACT_TOL)
    synth.check_numerics()


def test_images_vs_reference(synth, ka):
    from ganspace_b200.netdissect.nethook import InstrumentedModel
    z = torch.from_numpy(ka["z"]).cuda()
    with InstrumentedModel(synth) as inst:
        inst.retain_layer("g_synthesis.torgb")
        img = synth.forward(z)
        _check_known(ka, "torgb", inst.retained_layer("g_synthesis.torgb"), ACT_TOL)
    _check_known(ka, "img", img, IMG_TOL, grid=32)
    _check_known(ka, "mixed", synth.forward([z[:1]] * 8 + [z[1:2]] * 10), IMG_TOL, grid=32)
    synth.check_numerics()


def test_g_mapping_edit_strip_vs_reference(synth, ka):
    from ganspace_b200.netdissect.nethook import InstrumentedModel
    z = torch.from_numpy(ka["z"][:1]).cuda()
    d = torch.from_numpy(ka["strip_direction"]).cuda()
    s = torch.from_numpy(ka["strip_sigmas"]).cuda()
    with InstrumentedModel(synth) as inst:
        inst.edit_layer("g_mapping", offset=d[None, :] * s[:, None] * float(ka["strip_stdev"]))
        strip = synth.forward(z.repeat_interleave(5, dim=0))
    _check_known(ka, "strip", strip, IMG_TOL, grid=32)


def test_partial_equals_full_and_one_equals_eighteen(synth, ka):
    from ganspace_b200.netdissect.nethook import InstrumentedModel
    z = torch.from_numpy(ka["z"]).cuda()
    layers = ["g_synthesis.blocks.64x64", "g_synthesis.blocks.128x128.conv0_up", "g_synthesis.blocks.16x16.epi1.style_mod.lin"]
    with InstrumentedModel(synth) as inst:
        inst.retain_layers(layers)
        synth.partial_forward(z, "g_synthesis.blocks.128x128")
        part = {k: v.clone() for k, v in inst.retained_features().items()}
        img = synth.forward(z)
        full = inst.retained_features()
        for k in layers:
            assert torch.equal(part[k], full[k]), k
    assert torch.equal(img, synth.forward([z] * 18))
    # the decomposition's producer writes the same values in NHWC order, into a row-strided buffer
    buf = torch.zeros((2, 64 * 64 * 256 + 8), device="cuda")
    synth.activations_into(z, "g_synthesis.blocks.64x64", buf[:, :64 * 64 * 256])
    assert synth.feature_layout("g_synthesis.blocks.64x64") == ("nhwc", (64, 64, 256))
    assert torch.equal(buf[:, :64 * 64 * 256].view(2, 64, 64, 256).permute(0, 3, 1, 2), part["g_synthesis.blocks.64x64"])
    assert torch.count_nonzero(buf[:, 64 * 64 * 256:]) == 0


def test_unsupported_hooks_and_edits_raise(synth):
    from ganspace_b200.netdissect.nethook import InstrumentedModel
    z = synth.sample_latent(2, seed=3)
    for name in ("g_synthesis.blocks.8x8.epi1.top_epi.noise", "g_synthesis.blocks.4x4.epi1.top_epi.activation",
                 "g_synthesis.blocks.8x8.epi2.top_epi.instance_norm", "g_synthesis.blocks.16x16.conv0_up.upscale"):
        with InstrumentedModel(synth) as inst:
            inst.retain_layer(name)
            with pytest.raises(NotImplementedError, match=name.replace(".", r"\.")):
                synth.partial_forward(z, "g_synthesis.blocks.16x16")
    with InstrumentedModel(synth) as inst:
        inst.edit_layer("g_synthesis.blocks.8x8", offset=torch.ones(512, device="cuda"))
        with pytest.raises(NotImplementedError, match="cannot be propagated"):
            synth.partial_forward(z, "g_synthesis.blocks.16x16")
        with pytest.raises(NotImplementedError, match="cannot be propagated"):
            synth.forward(z)
    with pytest.raises(RuntimeError, match="not encountered in partial_forward"):
        synth.partial_forward(z, "g_synthesis.torgb")            # no block contains it (wrappers.py:417)
    synth.check_numerics()


def test_get_or_compute_synthesis_block_vs_reference(synth, golden, oracle):
    from ganspace_b200.config import Config
    from ganspace_b200.decomposition import get_or_compute
    from ganspace_b200.models import get_instrumented_model
    g = golden("sg1_ffhq_blocks8x8_z_n4000_b500_c4.npz")
    g["act_comp"] = g.pop("act_comp_f16").astype(np.float32)
    cfg = Config(output_class="ffhq", layer="g_synthesis.blocks.8x8", n=4_000, batch_size=500, components=4)
    inst = get_instrumented_model(cfg, torch.device("cuda:0"), model=synth)
    try:
        with tempfile.TemporaryDirectory() as tmp:
            path = get_or_compute(cfg, inst, submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp), force_recompute=True)
            with np.load(path, allow_pickle=False) as data:
                out = {k: data[k] for k in data.files}
    finally:
        inst.close()
    assert path.name == str(g["dump_name"])
    for k in ("act_comp", "act_mean", "act_stdev", "lat_comp", "lat_mean", "lat_stdev", "var_ratio", "random_stdevs"):
        assert out[k].shape == g[k].shape and out[k].dtype == np.float32, k
    cmp = oracle.compare_npz(out, g)
    assert cmp["min_signed_cos"] >= COS_TOL and cmp["min_lat_signed_cos"] >= COS_TOL, cmp
    assert cmp["max_abs_dvar_ratio"] <= RATIO_TOL, cmp
    for k in ("act_mean_rel", "act_stdev_rel", "lat_stdev_rel", "random_stdevs_rel"):
        assert cmp[k] < 10 * AUX_TOL, (k, cmp)
    synth.check_numerics()
