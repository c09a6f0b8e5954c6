"""ORACLE -- StyleGAN (v1) golden fixtures (tests/golden/), produced by the UNMODIFIED reference on CPU.

The reference is imported through oracle/ref_harness.py; the one override is ``rand_init_stylegan`` below, which replaces only
``load_model`` (checkpoint download / TF conversion, wrappers.py:311-345) by ``torch.manual_seed(seed); StyleGAN_G(res)``.

  sg1_mapping_known_answers.npz        (a) z = sample_latent(4, seed=...) in Z space, w = g_mapping(z) (wrappers.py:347-359),
                                           the output of g_mapping.dense3 (pre-activation) and of the shared dense*_act module
                                           (its last call) retained by hooks,
                                           the W-space sample_latent of the same seed, and the global-seed draw order
                                       (d) the reference's named_modules() list and per-parameter float64 sums, ffhq (1024^2)
                                           and bedrooms (256^2), random init seed 1234
  sg1_synthesis_known_answers.npz      (b) activations of two latents at 4x4, 8x8.conv0_up, 16x16.epi1, 64x64 (last nearest-upscale
                                           block), 128x128.conv0_up (first fused block), 1024x1024, 32x32.epi2.style_mod.lin and
                                           torgb (strided subsamples on a 16 x 16 raster + float64 sum / sum of squares)
                                       (c) images: forward(z) of the two latents, forward(18-list) with style mixing (8 + 10),
                                           and an offset edit strip on g_mapping (5 sigmas in [-2, 2] along a fixed direction);
                                           32 x 32 subsamples + sums
                                       with perturbed noise weights, conv biases, StyleMod biases and torgb bias (all zero at
                                       init; PERTURB below, recorded in the fixture) and noise seed 0
  sg1_ffhq_g_mapping_z_n10000_b1000_c32.npz   (e) get_or_compute(Config(output_class='ffhq'), n=10000, batch_size=1000, components=32),
                                                   Z space (PCA + latent regression)
  sg1_ffhq_g_mapping_w_n10000_b1000_c32.npz   (e) the same in W space (--use_w)
  sg1_ffhq_blocks8x8_z_n4000_b500_c4.npz      (e) layer g_synthesis.blocks.8x8 (d = 32768), Z space, n=4000, batch_size=500,
                                                   components=4, synthesis parameters perturbed as in (b); act_comp stored as
                                                   float16 (act_comp_f16) to keep the fixture small

Reference CPU time on the generator's host (torch 2.11 CPU, all cores): (a)+(d) 4 s, (b)+(c) 7 s, each
g_mapping (e) run 2-5 s, the 8x8 block (e) run 53 s.

Usage:  python oracle/gen_golden_sg1.py [a] [b] [e] [e8]   (a: (a)+(d), b: (b)+(c), e / e8: (e); default all)
"""
import sys
import tempfile
import time
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
from oracle import ref_harness as rh          # noqa: E402

OUT = REPO / "tests" / "golden"
SEED_INIT = 1234


def rand_init_stylegan(ref, device, outclass="ffhq", seed=SEED_INIT):
    """The reference's StyleGAN wrapper with random-init weights (load_model is the only override)."""

    class RandInitStyleGAN(ref.wrappers.StyleGAN):
        def load_model(self):
            torch.manual_seed(seed)
            self.model = ref.wrappers.stylegan.StyleGAN_G(self.resolution).to(self.device)

    return RandInitStyleGAN(device, outclass)


def known_answers():
    ref = rh.import_reference()
    dev = torch.device("cpu")
    ka = {}
    for outclass in ("ffhq", "bedrooms"):
        m = rand_init_stylegan(ref, dev, outclass)
        names = [n for n, _ in m.model.named_modules()]
        params = list(m.model.named_parameters())
        ka[f"{outclass}_module_names"] = np.array(names)
        ka[f"{outclass}_param_names"] = np.array([n for n, _ in params])
        ka[f"{outclass}_param_sums"] = np.array([p.detach().double().sum().item() for _, p in params])
        ka[f"{outclass}_param_abs_sums"] = np.array([p.detach().double().abs().sum().item() for _, p in params])
        ka[f"{outclass}_buffer_names"] = np.array([n for n, _ in m.model.named_buffers()])
    m = rand_init_stylegan(ref, dev, "ffhq")
    mapping = m.model._modules["g_mapping"]
    with torch.no_grad():
        m.use_z()
        z = m.sample_latent(4, seed=77)
        ka["z"] = z.numpy()
        ka["w"] = mapping.forward(z).numpy()
        # a dense layer and the shared activation module, retained through the reference's own hooks (nethook)
        from netdissect.nethook import InstrumentedModel
        inst = InstrumentedModel(m)
        inst.retain_layers(["g_mapping.dense3", "g_mapping.dense0_act"])
        m.partial_forward(z, "g_mapping")
        ka["dense3"] = inst.retained_layer("g_mapping.dense3").numpy()
        ka["dense0_act_last"] = inst.retained_layer("g_mapping.dense0_act").numpy()   # the last of its 8 calls = w
        inst.close()
        m.use_w()
        ka["w_sample_seed77"] = m.sample_latent(4, seed=77).numpy()
        # sample_latent() without a seed: the global NumPy state decides (wrappers.py:348-349)
        np.random.seed(5)
        m.use_z()
        ka["z_global_seed5"] = m.sample_latent(2).numpy()
    np.savez_compressed(OUT / "sg1_mapping_known_answers.npz", **ka)
    print("wrote sg1_mapping_known_answers.npz")


def decomposition(use_w, n=10_000, b=1_000, c=32, layer=None, out_name=None, f16_comp=False):
    ref = rh.import_reference()
    dev = torch.device("cpu")
    m = rand_init_stylegan(ref, dev, "ffhq")
    # Config()'s model / layer / estimator defaults; its output_class default (None) names no StyleGAN class, and the
    # reference's get_or_compute needs one for the cache name (decomposition.py:386)
    cfg = ref.Config(output_class="ffhq", n=n, batch_size=b, components=c, use_w=use_w)
    assert (cfg.model, cfg.layer, cfg.output_class, cfg.estimator) == ("StyleGAN", "g_mapping", "ffhq", "ipca")
    if layer is not None:
        cfg.layer = layer
        perturb_synthesis(m.model)
        m.set_noise_seed(0)
    inst = ref.wrappers.get_instrumented_model(cfg, dev, model=m)
    t0 = time.time()
    with tempfile.TemporaryDirectory() as tmp:
        path = ref.decomposition.get_or_compute(cfg, inst, force_recompute=True,
                                                submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp))
        with np.load(path) as data:
            out = {k: data[k].copy() for k in data.files}
        name = path.name
    print(f"{cfg.layer} use_w={use_w}: {time.time() - t0:.1f} s -> {name}", flush=True)
    inst.close()
    tag = "w" if use_w else "z"
    out_name = out_name or f"sg1_ffhq_g_mapping_{tag}_n{n}_b{b}_c{c}.npz"
    if f16_comp:
        out["act_comp_f16"] = out.pop("act_comp").astype(np.float16)
    np.savez_compressed(OUT / out_name, dump_name=np.array(name), **out)


PERTURB = 0.2          # scale of the standard-normal values written into the zero-initialised synthesis parameters
KA_LAYERS = ["g_synthesis.blocks.4x4", "g_synthesis.blocks.8x8.conv0_up", "g_synthesis.blocks.16x16.epi1",
             "g_synthesis.blocks.64x64", "g_synthesis.blocks.128x128.conv0_up", "g_synthesis.blocks.1024x1024",
             "g_synthesis.blocks.32x32.epi2.style_mod.lin", "g_synthesis.torgb"]


def perturb_synthesis(G, seed=9):
    """Non-zero noise weights, conv biases, StyleMod biases and torgb bias (zero at random init) from a fixed generator; the
    InputBlock bias (init 1) and the const are left as they are."""
    g = torch.Generator().manual_seed(seed)
    names = []
    with torch.no_grad():
        for k, p in G.named_parameters():
            if k.startswith("g_synthesis") and (k.endswith("noise.weight") or (k.endswith(".bias") and not k.endswith("4x4.bias"))):
                p.copy_(PERTURB * torch.randn(p.shape, generator=g))
                names.append(k)
    return names


def _known(ka, key, act, grid=16):
    """float64 sum / sum of squares of the whole activation and a strided subsample: every (C // 16)-th channel on a
    grid x grid raster (images: grid 32)."""
    act = np.asarray(act)
    ka[f"sum_{key}"] = np.array([act.astype(np.float64).sum(), (act.astype(np.float64) ** 2).sum()])
    ka[f"shape_{key}"] = np.array(act.shape)
    if act.ndim == 4:
        step = max(1, act.shape[-1] // grid)
        act = act[:, ::max(1, act.shape[1] // 16), ::step, ::step]
    ka[f"act_{key}_sub"] = act.copy()


def synthesis_known_answers():
    ref = rh.import_reference()
    from netdissect.nethook import InstrumentedModel      # the reference's (importable once import_reference ran)
    dev = torch.device("cpu")
    m = rand_init_stylegan(ref, dev, "ffhq")
    perturbed = perturb_synthesis(m.model)
    m.set_noise_seed(0)
    m.use_z()
    z = m.sample_latent(2, seed=21)
    ka = dict(z=z.numpy(), layers=np.array(KA_LAYERS), perturbed=np.array(perturbed), perturb_scale=np.array(PERTURB))
    t0 = time.time()
    inst = InstrumentedModel(m)
    inst.retain_layers(KA_LAYERS)
    with torch.no_grad():
        img = m.forward(z).numpy()
    for layer in KA_LAYERS:
        _known(ka, layer.replace("g_synthesis.", "").replace(".", "_"), inst.retained_layer(layer).numpy())
    inst.close()
    # control: partial_forward gives the same block output as the full forward
    inst = InstrumentedModel(m)
    inst.retain_layer("g_synthesis.blocks.64x64")
    with torch.no_grad():
        m.partial_forward(z, "g_synthesis.blocks.64x64")
    a = inst.retained_layer("g_synthesis.blocks.64x64").numpy()
    assert np.array_equal(a[:, ::16, ::4, ::4], ka["act_blocks_64x64_sub"])
    inst.close()
    with torch.no_grad():
        mixed = m.forward([z[:1]] * 8 + [z[1:2]] * 10).numpy()
        same = m.forward([z[:1]] * 18).numpy()
    assert np.abs(same - img[:1]).max() < 1e-4 * np.abs(img).max(), np.abs(same - img[:1]).max()     # batch-size-dependent CPU conv order
    _known(ka, "img", img, grid=32)
    _known(ka, "mixed", mixed, grid=32)
    # an 'activation'-mode edit strip on g_mapping (the notebooks' _create_strip_batch_sigma, centre=False): one latent
    # repeated 5 times, offset sigma * stdev * direction on the g_mapping output
    g = torch.Generator().manual_seed(31)
    direction = torch.randn(512, generator=g)
    direction = direction / direction.norm()
    sigmas = torch.linspace(-2.0, 2.0, 5)
    offset = direction[None, :] * sigmas[:, None] * 0.7
    inst = InstrumentedModel(m)
    inst.edit_layer("g_mapping", offset=offset)
    with torch.no_grad():
        strip = m.forward(z[:1].repeat_interleave(5, dim=0)).numpy()
    inst.close()
    ka.update(strip_direction=direction.numpy(), strip_sigmas=sigmas.numpy(), strip_stdev=np.array(0.7))
    _known(ka, "strip", strip, grid=32)
    print(f"synthesis known answers: {time.time() - t0:.0f} s")
    np.savez_compressed(OUT / "sg1_synthesis_known_answers.npz", **ka)


if __name__ == "__main__":
    which = set(sys.argv[1:]) or {"a", "b", "e"}
    if "a" in which:
        known_answers()
    if "b" in which:
        synthesis_known_answers()
    if "e" in which:
        decomposition(False)
        decomposition(True)
    if "e8" in which or not sys.argv[1:]:
        decomposition(False, 4_000, 500, 4, layer="g_synthesis.blocks.8x8", out_name="sg1_ffhq_blocks8x8_z_n4000_b500_c4.npz",
                      f16_comp=True)
