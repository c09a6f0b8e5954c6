"""Model wrappers of the hot path: ``BaseModel``, ``StyleGAN2``, ``get_model``, ``get_instrumented_model``.

Mirror of /root/reference/models/wrappers.py (BaseModel :27-94, StyleGAN2 :97-267, factories :651-735):
same class and method names, argument meaning and error behaviour, so ``decomposition.get_or_compute``,
``visualize.py`` and the notebooks call them unchanged.  Differences, all on the device side:

* ``sample_latent`` draws the NumPy-legacy normal stream ON THE GPU (bit-exact MT19937 + polar method,
  csrc/rng.cu) -- the seed is still taken from NumPy's global state on the host exactly as the reference
  does (wrappers.py:168-169), so seeds and latents are identical.
* ``Generator.style`` runs the hand-written mapping kernels (csrc/mapping*.cu).
* ``partial_forward(x, 'style')`` stops right after the mapping network; the reference first builds the
  ``[B, n_latent, 512]`` repeat+stack that the early exit then throws away (wrappers.py:202-222).
* checkpoints: no network here.  A rosinality ``g_ema`` checkpoint under $GANCONTROL_CHECKPOINT_DIR is
  loaded when present; otherwise ``random_init=<seed>`` (or env GANSPACE_B200_RANDOM_INIT) reproduces the
  reference's default initialisation under ``torch.manual_seed(seed)`` (the BASELINE.json configs).
"""
from __future__ import annotations

import os
from abc import ABC as AbstractBaseClass, abstractmethod
from functools import singledispatch
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

from .. import _native
from ..config import Config
from ..netdissect.nethook import InstrumentedModel
from . import stylegan, stylegan2

INT32_MAX = int(np.iinfo(np.int32).max)


def _global_seed() -> int:
    """``np.random.randint(np.iinfo(np.int32).max)`` on NumPy's global legacy state (wrappers.py:169)."""
    return int(np.random.randint(INT32_MAX))


def _checkpoint_or_seed(family, rel_path, random_init):
    """(checkpoint path, random-init seed or None).  The seed is ``random_init``, else env GANSPACE_B200_RANDOM_INIT; without
    one the checkpoint under $GANCONTROL_CHECKPOINT_DIR must exist (there is no download)."""
    root = os.environ.get("GANCONTROL_CHECKPOINT_DIR", Path(__file__).parent / "checkpoints")
    checkpoint = Path(root) / rel_path
    seed = random_init
    if seed is None and os.environ.get("GANSPACE_B200_RANDOM_INIT"):
        seed = int(os.environ["GANSPACE_B200_RANDOM_INIT"])
    if seed is None and not checkpoint.is_file():
        raise RuntimeError(
            f"{family} checkpoint {checkpoint} not found and no network access to download it; pass "
            "random_init=<seed> (or set GANSPACE_B200_RANDOM_INIT) for random-init weights")
    return checkpoint, seed


class BaseModel(AbstractBaseClass, torch.nn.Module):
    def __init__(self, model_name, class_name):
        super().__init__()
        self.model_name = model_name
        self.outclass = class_name

    @abstractmethod
    def partial_forward(self, x, layer_name):
        """Run the network only up to ``layer_name`` (hooks fire as a side effect); returns None."""

    @abstractmethod
    def sample_latent(self, n_samples=1, seed=None, truncation=None):
        """Batch of latents on ``self.device``."""

    def get_max_latents(self):
        return 1

    def latent_space_name(self):
        return "Z"

    def get_latent_shape(self):
        return tuple(self.sample_latent(1).shape)

    def get_latent_dims(self):
        return np.prod(self.get_latent_shape())

    def set_output_class(self, new_class):
        self.outclass = new_class

    def forward(self, x):
        out = self.model.forward(x)
        return 0.5 * (out + 1)

    def sample_np(self, z=None, n_samples=1, seed=None):
        if z is None:
            z = self.sample_latent(n_samples, seed=seed)
        elif isinstance(z, list):
            z = [torch.tensor(l).to(self.device) if not torch.is_tensor(l) else l for l in z]
        elif not torch.is_tensor(z):
            z = torch.tensor(z).to(self.device)
        img = self.forward(z)
        img_np = img.permute(0, 2, 3, 1).cpu().detach().numpy()
        return np.clip(img_np, 0.0, 1.0).squeeze()

    def get_conditional_state(self, z):
        return None

    def set_conditional_state(self, z, c):
        return z

    def named_modules(self, *args, **kwargs):
        return self.model.named_modules(*args, **kwargs)


class _MappedLatentModel(BaseModel):
    """What StyleGAN and StyleGAN2 share (wrappers.py:167-179, :302-309, :347-366): Z drawn from the NumPy-legacy stream on the
    device, W = the mapping network (``_mapping_net()``, a module with ``packed()``) applied to it, and the producer
    interface the decomposition driver uses (``sample_latents_multi``, ``draw_z_async``, ``z_to_latent``,
    ``check_numerics``)."""

    def _mapping_net(self):
        raise NotImplementedError

    def latent_space_name(self):
        return "W" if self.w_primary else "Z"

    def use_w(self):
        self.w_primary = True

    def use_z(self):
        self.w_primary = False

    def set_output_class(self, new_class):
        if self.outclass != new_class:
            raise RuntimeError(f"{self.model_name}: cannot change output class without reloading")

    def get_latent_shape(self):
        """The reference samples one latent for its shape (wrappers.py:60-61).  The draw from the global NumPy stream that this
        sample_latent(1) consumes is kept (later seeds depend on it); the two kernels behind it are not launched."""
        _global_seed()
        return (1, 512)

    def sample_latent(self, n_samples=1, seed=None, truncation=None):
        if seed is None:
            seed = _global_seed()
        z = _native.legacy_normal([seed], 512 * n_samples, self.device).view(n_samples, 512)
        if self.w_primary:
            z = self._mapping_net()(z)
        return z

    def draw_z_async(self, n_samples, seed):
        """The Z stream of ``sample_latent(n_samples, seed=seed)`` generated on a side stream; returns a callable that makes
        the current stream wait for it and hands back z [n_samples, 512]."""
        side = getattr(self, "_side_stream", None)
        if side is None:
            with torch.cuda.device(self.device):
                side = self._side_stream = torch.cuda.Stream(device=self.device)
        with torch.cuda.device(self.device):
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                z = _native.legacy_normal([seed], 512 * n_samples, self.device).view(n_samples, 512)

        def result():
            with torch.cuda.device(self.device):
                torch.cuda.current_stream().wait_stream(side)
            z.record_stream(torch.cuda.current_stream())
            return z
        return result

    def z_to_latent(self, z):
        """What sample_latent does after drawing z (wrappers.py:176-179): the mapping network in W mode."""
        return self._mapping_net()(z) if self.w_primary else z

    def sample_latents_multi(self, n_samples, seeds, out=None, lazy=False):
        """Several ``sample_latent(n_samples, seed=s)`` calls in ONE launch (one CTA per seed);
        ``out`` is an optional [len(seeds)*n_samples, 512] device buffer.  Used by the decomposition
        driver so that a whole run's ~100 independent streams fill the machine.
        ``lazy=True`` (W space): returns (z, ensure) where ``ensure(row_end)`` maps rows [0, row_end) to W in
        place, chunk by chunk, so that the consumer of the first rows does not wait for the last ones."""
        S = len(seeds)
        parts = _native.split_parts(512 * n_samples)
        if not lazy:
            z = _native.legacy_normal(list(seeds), 512 * n_samples, self.device,
                                      out=None if out is None else out.view(S, 512 * n_samples), parts=parts)
            z = z.view(S * n_samples, 512)
            if not self.w_primary:
                return z
            return self._mapping_net()(z) if out is None else self._mapping_net().packed().forward(z, out=z)
        # lazy: the streams are generated in launch groups on a side stream (a small first group, so that the first
        # partial_fit group exists after ~1.5 ms instead of after the whole run's RNG); ensure(row_end) waits for the groups
        # that cover rows [0, row_end) and, in W mode, maps them group by group in place.
        z = torch.empty((S * n_samples, 512), dtype=torch.float32, device=self.device) if out is None else out.view(S * n_samples, 512)
        # group sizes in streams (x parts CTAs each).  Measured (tools/phase_probe.py, config 2): the merge chain's 16-CTA cluster
        # launches need free SMs at every step, so the producers share the machine statically -- 7 streams x 8 = 56 RNG CTAs,
        # 76 persistent GEMM CTAs (GANSPACE_B200_LAZY_FREE_SMS = 72), 16 SMs for the chain
        sizes = [int(v) for v in os.environ.get("GANSPACE_B200_RNG_GROUPS", "4,7").split(",")]
        bounds, g0 = [], 0
        while g0 < S:
            g1 = min(S, g0 + sizes[min(len(bounds), len(sizes) - 1)])
            bounds.append((g0, g1))
            g0 = g1
        sides = getattr(self, "_rng_streams", None)
        if sides is None:                       # (more than one stream: groups alternate; measured slower -- they crowd out the GEMMs)
            with torch.cuda.device(self.device):
                sides = self._rng_streams = [torch.cuda.Stream(device=self.device)
                                             for _ in range(max(1, int(os.environ.get("GANSPACE_B200_RNG_STREAMS", "1"))))]
        events = []
        seeds_dev = _native.seeds_tensor(list(seeds), self.device)       # ONE host->device copy, before any long kernel is queued
        # the first group decides when the first partial_fit statistics exist (the merge chain, the critical path of a small-d
        # run, waits for them): its streams are split over twice as many CTAs (GANSPACE_B200_RNG_FIRST_PARTS)
        parts0 = parts
        if parts > 1:
            parts0 = max(parts, min(16, int(os.environ.get("GANSPACE_B200_RNG_FIRST_PARTS", 2 * parts))))
            _native.jump_polys(512 * n_samples, parts, self.device)     # (first use: host computation + upload)
            _native.jump_polys(512 * n_samples, parts0, self.device)
            # one scratch buffer for the largest group, so that no launch re-allocates it while an earlier one is running
            gmax = max(b - a for a, b in bounds)
            wsb = _native.load().gsb_legacy_normal_split_workspace_bytes
            need = max(wsb(gmax, 512 * n_samples, parts), wsb(bounds[0][1] - bounds[0][0], 512 * n_samples, parts0))
            for i, side in enumerate(sides):
                _native.scratch.get(f"rng_split{i}", need, _native.require_cuda(self.device)).record_stream(side)
        with torch.cuda.device(self.device):
            for side in sides:
                side.wait_stream(torch.cuda.current_stream())
            for gi, (a, b) in enumerate(bounds):
                side = sides[gi % len(sides)]
                with torch.cuda.stream(side):
                    _native.legacy_normal(seeds_dev[a:b], 512 * n_samples, self.device,
                                          out=z[a * n_samples:b * n_samples].view(b - a, 512 * n_samples),
                                          parts=parts0 if gi == 0 else parts, scratch_key=f"rng_split{gi % len(sides)}")
                    ev = torch.cuda.Event()
                    ev.record(side)
                    events.append(ev)
            for side in sides:
                z.record_stream(side)
                seeds_dev.record_stream(side)          # read by launches that run long after this function has returned
        packed = self._mapping_net().packed() if self.w_primary else None
        state = {"g": 0, "keep": seeds_dev}
        free_sms = int(os.environ.get("GANSPACE_B200_LAZY_FREE_SMS", 72 if parts > 1 else 48))

        def ensure(row_end):
            # later groups run next to the IPCA chain and leave a GPC's worth of SMs to it
            while state["g"] < len(bounds) and bounds[state["g"]][0] * n_samples < row_end:
                g = state["g"]
                a, b = bounds[g][0] * n_samples, bounds[g][1] * n_samples
                torch.cuda.current_stream().wait_event(events[g])
                if packed is not None:
                    packed.forward(z[a:b], out=z[a:b], leave_free_sms=0 if g == 0 else free_sms)
                state["g"] = g + 1
        return z, ensure

    def check_numerics(self):
        """Raise if a kernel flagged an out-of-range activation since the weights were packed (synchronises)."""
        self._mapping_net().packed().check()
        if getattr(self, "_synth_cache", None) is not None:
            self._synth_cache[1].check()


class StyleGAN2(_MappedLatentModel):
    CONFIGS = {"ffhq": 1024, "car": 512, "cat": 256, "church": 256, "horse": 256,
               "bedrooms": 256, "kitchen": 256, "places": 256}

    def __init__(self, device, class_name, truncation=1.0, use_w=False, random_init=None):
        super().__init__("StyleGAN2", class_name or "ffhq")
        self.device = _native.require_cuda(device)
        self.truncation = truncation
        self.latent_avg = None
        self.w_primary = use_w
        assert self.outclass in self.CONFIGS, \
            f'Invalid StyleGAN2 class {self.outclass}, should be one of [{", ".join(self.CONFIGS.keys())}]'
        self.resolution = self.CONFIGS[self.outclass]
        self.name = f"StyleGAN2-{self.outclass}"
        self.has_latent_residual = True
        self._random_init = random_init
        self.load_model()
        self.set_noise_seed(0)

    def _mapping_net(self):
        return self.model.style

    def load_model(self):
        checkpoint, seed = _checkpoint_or_seed("StyleGAN2", f"stylegan2/stylegan2_{self.outclass}_{self.resolution}.pt",
                                               self._random_init)
        if seed is None:
            self.model = stylegan2.Generator(self.resolution, 512, 8)
            ckpt = torch.load(checkpoint, map_location="cpu")
            self.model.load_state_dict(ckpt["g_ema"], strict=False)
            self.model = self.model.to(self.device)
            self.latent_avg = ckpt["latent_avg"].to(self.device)
        else:
            # the reference's default init, bit-for-bit: parameters are created on the host in the
            # reference's order under one manual seed, then moved to the device
            torch.manual_seed(int(seed))
            self.model = stylegan2.Generator(self.resolution, 512, 8).to(self.device)
            self.latent_avg = torch.zeros(512, device=self.device)

    def get_max_latents(self):
        return self.model.n_latent

    def forward(self, x):
        """wrappers.py:188-192: images in [0, 1] (before clamping) from one latent, a pair, or one latent per layer.  Hooked
        StyledConv / ToRGB layers receive their activations (retain_layer works); an edit installed on a hooked layer would
        have to be re-fed into the fused chain, which is not built -- it raises instead of being silently ignored."""
        x = x if isinstance(x, list) else [x]
        names = self.synthesis_layer_names()
        syn = self._synthesis(len(names))
        out, latent = self.model(x, noise=self.noise, truncation=self.truncation, truncation_latent=self.latent_avg,
                                 input_is_w=self.w_primary, return_latents=True, _synthesis=syn)
        self._fire_hooks(latent, len(names) - 1, rgb_upto=len(self.model.to_rgbs))
        return 0.5 * (out + 1)

    def _fire_hooks(self, latent, target, rgb_upto=-1):
        """Hand the activations of hooked StyledConv layers 0..target (and hooked ToRGB layers 0..rgb_upto) to their hooks:
        each gets its own run of the fused chain up to that layer."""
        mods = [self.model.conv1] + list(self.model.convs)
        rgbs = [self.model.to_rgb1] + list(self.model.to_rgbs)
        w_layers = latent.permute(1, 0, 2).contiguous()
        for i in range(target + 1):
            if len(mods[i]._forward_hooks):
                syn = self._synthesis(i + 1)
                res, co = syn.shapes[i]
                act, _ = syn.render(w_layers, i + 1, [], want_act=True)
                act = act.view(-1, res, res, co).permute(0, 3, 1, 2)                   # NCHW view of NHWC storage
                if mods[i](_result=act) is not act:
                    raise NotImplementedError(f"an edit on layer '{self.synthesis_layer_names()[i]}' cannot be propagated through "
                                              "the fused synthesis chain")
        for j in range(rgb_upto + 1):
            if len(rgbs[j]._forward_hooks):
                syn = self._synthesis(2 * j + 1)
                _, img = syn.render(w_layers, 2 * j + 1, [r.describe() for r in rgbs[:j + 1]])
                img = img.permute(0, 3, 1, 2)
                if rgbs[j](_result=img) is not img:
                    raise NotImplementedError("an edit on a ToRGB layer cannot be propagated through the fused synthesis chain")

    # ---- synthesis chain conv1, convs.0 .. convs.k (wrappers.py:224-255) ------------------------------------
    def synthesis_layer_names(self):
        return ["conv1"] + [f"convs.{i}" for i in range(len(self.model.convs))]

    def _synthesis(self, n_run):
        """PackedSynthesis covering at least the first ``n_run`` StyledConv layers (re-packed when a parameter or a
        noise map of those layers changes, or when a deeper layer is asked for)."""
        mods = [self.model.conv1] + list(self.model.convs)
        cst = self.model.input.input
        keys = [(cst._version, cst.data_ptr())]
        keys += [(m.conv.weight._version, m.conv.weight.data_ptr(), m.conv.modulation.weight._version,
                  m.conv.modulation.bias._version, m.noise.weight._version, m.activate.bias._version,
                  self.noise[i].data_ptr(), self.noise[i]._version) for i, m in enumerate(mods[:n_run])]
        cached = getattr(self, "_synth_cache", None)
        if cached is None or len(cached[0]) < len(keys) or cached[0][:len(keys)] != keys:
            layers, res = [], 4
            for i, m in enumerate(mods[:n_run]):
                layers.append(m.describe(self.noise[i], res))
                res = 2 * res if m.conv.upsample else res
            packed = _native.PackedSynthesis(cst.detach()[0], layers, self.model.style_dim)
            self._synth_cache = cached = (keys, packed)
        return cached[1]

    def feature_layout(self, layer_name):
        """Native (device) feature order of ``activations_into`` for this layer: ('nhwc', (H, W, C)); the reference's
        flattening is NCHW -- a fixed permutation, applied once to the exported components."""
        names = self.synthesis_layer_names()
        if layer_name not in names:
            return None
        res, co = self._synthesis(names.index(layer_name) + 1).shapes[names.index(layer_name)]
        return ("nhwc", (res, res, co))

    def activations_into(self, x, layer_name, out):
        """Hooked-layer activations of latents x [n,512] (in the current primary space) written as fp32 NHWC rows into
        ``out`` [n, H*W*C] (may be row-strided): the decomposition driver's producer for conv layers."""
        names = self.synthesis_layer_names()
        n_run = names.index(layer_name) + 1
        w = x if self.w_primary else self.model.style(x)
        return self._synthesis(n_run).forward(w.reshape(-1, 512), n_run, out=out)

    def partial_forward(self, x, layer_name):
        """wrappers.py:194-259: run up to (and including) the named layer; side effect = its hooks fire.  ``x``: one latent, a
        pair (style mixing at a random index, as the reference) or one latent per layer."""
        styles = x if isinstance(x, list) else [x]
        if not self.w_primary:
            styles = [self.model.style(s) for s in styles]
        if "style" in layer_name:
            # (the reference builds the [N, n_latent, 512] repeat + StridedStyle stack before this early exit, wrappers.py:202-222 --
            # 328 MB of traffic per 10k batch that nothing reads; skipped here)
            return
        latent = self.model.latents_per_layer(styles)             # [N, n_latent, 512]
        if layer_name == "input":
            self.model.input(latent[:, 0])
            return
        names = self.synthesis_layer_names()
        rgb_names = ["to_rgb1"] + [f"to_rgbs.{i}" for i in range(len(self.model.to_rgbs))]
        rgb_hooked = any(len(m._forward_hooks) for m in [self.model.to_rgb1] + list(self.model.to_rgbs))
        if layer_name in names and len(styles) == 1 and not rgb_hooked:
            # one global latent, no ToRGB hook: the decomposition's own call pattern -- the single-latent entry point
            mods = [self.model.conv1] + list(self.model.convs)
            target = names.index(layer_name)
            w = styles[0].reshape(-1, 512)
            for i in [i for i in range(target) if len(mods[i]._forward_hooks)] + [target]:
                syn = self._synthesis(target + 1)
                res, co = syn.shapes[i]
                act = syn.forward(w, i + 1).view(-1, res, res, co).permute(0, 3, 1, 2)    # NCHW view of NHWC storage
                if mods[i](_result=act) is not act and i < target:
                    # (an edit on the target layer itself has nothing downstream inside partial_forward)
                    raise NotImplementedError(f"an edit on layer '{names[i]}' cannot be propagated through the fused synthesis "
                                              f"chain to '{layer_name}'")
        elif layer_name in names:
            target = names.index(layer_name)
            # the reference computes every to_rgb that precedes the target as well (wrappers.py:232-255)
            self._fire_hooks(latent, target, rgb_upto=(target - 1) // 2 if target >= 1 else -1)
        elif layer_name in rgb_names:
            j = rgb_names.index(layer_name)
            self._fire_hooks(latent, 2 * j, rgb_upto=j)
        else:
            raise RuntimeError(f"Unknown layer '{layer_name}'")

    def set_noise_seed(self, seed):
        # same generator stream as the reference (torch.manual_seed(seed); torch.randn per noise map),
        # drawn on the host so that it does not depend on the device RNG implementation
        torch.manual_seed(seed)
        self.noise = [torch.randn(1, 1, 2 ** 2, 2 ** 2).to(self.device)]
        for i in range(3, self.model.log_size + 1):
            for _ in range(2):
                self.noise.append(torch.randn(1, 1, 2 ** i, 2 ** i).to(self.device))


class StyleGAN(_MappedLatentModel):
    """wrappers.py:269-436 (StyleGAN 1, ``models/stylegan/model.py``).  The mapping network ``g_mapping`` runs on the packed
    mapping kernels and the synthesis network as one fused C-ABI call (models/stylegan.py, csrc/synthesis_sg1.cu).  Hooks on
    g_mapping retain and edit (the wrapper calls the module, so what its hooks return is what synthesis consumes).  Hooks on
    the synthesis stop points (blocks, epi1 / epi2, style_mod, style_mod.lin, conv / conv0_up / conv1, torgb, g_synthesis)
    receive their activations; an edit there would have to be re-fed into the fused chain, which is not built, and raises.  A
    hook on any other synthesis module (noise, activation, instance_norm, upscale, blur) raises NotImplementedError."""
    CONFIGS = {"ffhq": 1024, "celebahq": 1024, "bedrooms": 256, "cars": 512, "cats": 256, "vases": 1024, "wikiart": 512,
               "fireworks": 512, "abstract": 512, "anime": 512, "ukiyo-e": 512}

    def __init__(self, device, class_name, truncation=1.0, use_w=False, random_init=None):
        super().__init__("StyleGAN", class_name or "ffhq")
        self.device = _native.require_cuda(device)
        self.w_primary = use_w
        assert self.outclass in self.CONFIGS, \
            f'Invalid StyleGAN class {self.outclass}, should be one of [{", ".join(self.CONFIGS.keys())}]'
        self.resolution = self.CONFIGS[self.outclass]
        self.name = f"StyleGAN-{self.outclass}"
        self.has_latent_residual = True
        self._random_init = random_init
        self.load_model()
        self.set_noise_seed(0)
        self._stop_points = self._make_stop_points()

    def _mapping_net(self):
        return self.model.g_mapping

    def load_model(self):
        checkpoint, seed = _checkpoint_or_seed("StyleGAN", f"stylegan/stylegan_{self.outclass}_{self.resolution}.pt",
                                               self._random_init)
        if seed is None:
            self.model = stylegan.StyleGAN_G(self.resolution)
            self.model.load_state_dict(torch.load(checkpoint, map_location="cpu"))
            self.model = self.model.to(self.device)
        else:
            # the reference's default init, bit-for-bit (parameters created on the host under one manual seed)
            torch.manual_seed(int(seed))
            self.model = stylegan.StyleGAN_G(self.resolution).to(self.device)

    def get_max_latents(self):
        return 18

    # ---- the fused synthesis chain ------------------------------------------------------------------------
    def _make_stop_points(self):
        """module name -> (chain layer, stop) for every module whose output the chain can stop at.  Block i is chain layers
        2i (4x4: const + bias -> epi1; else conv0_up -> epi1) and 2i + 1 (conv / conv1 -> epi2)."""
        pts = {}
        blocks = list(self.model.g_synthesis.blocks.keys())
        for i, name in enumerate(blocks):
            pre = f"g_synthesis.blocks.{name}"
            pts[pre] = (2 * i + 1, "epi")
            for k, j in (("epi1", 2 * i), ("epi2", 2 * i + 1)):
                pts[f"{pre}.{k}"] = pts[f"{pre}.{k}.style_mod"] = (j, "epi")
                pts[f"{pre}.{k}.style_mod.lin"] = (j, "style")
            if i == 0:
                pts[f"{pre}.conv"] = (1, "conv")
            else:
                pts[f"{pre}.conv0_up"] = (2 * i, "conv")
                pts[f"{pre}.conv1"] = (2 * i + 1, "conv")
        pts["g_synthesis.torgb"] = pts["g_synthesis"] = (2 * len(blocks) - 1, "image")
        return pts

    def _synthesis(self):
        """PackedSG1 of the whole synthesis network, re-packed when a parameter or a noise map changes."""
        G = self.model.g_synthesis
        noises = [m.noise for m in G.modules() if isinstance(m, stylegan.NoiseLayer)]
        keys = (self._noise_generation,) + tuple((p._version, p.data_ptr()) for p in G.parameters()) + \
            tuple((t._version, t.data_ptr()) for t in noises)
        cached = getattr(self, "_synth_cache", None)
        if cached is None or cached[0] != keys:
            def epi(e):
                return dict(noise_weight=e.top_epi.noise.weight, noise=e.top_epi.noise.noise, style_weight=e.style_mod.lin.weight,
                            style_bias=e.style_mod.lin.bias)
            layers = []
            for i, (name, blk) in enumerate(G.blocks.items()):
                res = int(name.split("x")[0])
                if i == 0:
                    c = blk.nf
                    layers.append(dict(kind="const", weight=blk.const[0], bias=blk.bias, cin=c, cout=c, res_out=4, **epi(blk.epi1)))
                    layers.append(dict(kind="same", weight=blk.conv.weight, bias=blk.conv.bias, cin=c, cout=c, res_out=4,
                                       **epi(blk.epi2)))
                else:
                    # model.py:82: the fused transposed conv from 128^2 on, nearest upscale + conv below
                    co, ci = blk.conv0_up.weight.shape[:2]
                    layers.append(dict(kind="fused" if res >= 128 else "nearest", weight=blk.conv0_up.weight, bias=blk.conv0_up.bias,
                                       cin=ci, cout=co, res_out=res, **epi(blk.epi1)))
                    layers.append(dict(kind="same", weight=blk.conv1.weight, bias=blk.conv1.bias, cin=co, cout=co, res_out=res,
                                       **epi(blk.epi2)))
            packed = _native.PackedSG1(layers, G.torgb.weight[:, :, 0, 0], G.torgb.bias, G.dlatent_size)
            self._synth_cache = cached = (keys, packed)
        return cached[1]

    def _latents(self, x):
        """[Lw, n, 512] per-layer W latents (Lw = 1: one latent for every layer) from one latent or a list of 18
        (wrappers.py:378-385, model.py:376-385); in Z space through the g_mapping module, so its hooks fire and edit."""
        if isinstance(x, list):
            assert len(x) == 18, "Must provide 1 or 18 latents"
            ws = x if self.w_primary else [self.model.g_mapping(l) for l in x]
            return torch.stack([w.reshape(-1, 512) for w in ws], dim=0)
        w = x if self.w_primary else self.model.g_mapping(x)
        return w.reshape(1, -1, 512)

    def _run(self, w_layers, point):
        j, stop = point
        syn = self._synthesis()
        n = w_layers.shape[1]
        out = syn.forward(w_layers, j + 1, stop)
        if stop == "style":
            return out
        res, co = syn.shapes[j]
        if stop == "image":
            return out.view(n, 3, res, res)
        return out.view(n, res, res, co).permute(0, 3, 1, 2)                 # NCHW view of NHWC storage

    def _fire_hooks(self, w_layers, modules):
        """Hand every hooked module of ``modules`` (name, module) its output, each from its own run of the chain."""
        for name, m in modules:
            if not (len(m._forward_hooks) or len(m._forward_pre_hooks)):
                continue
            point = self._stop_points.get(name)
            if point is None:
                raise NotImplementedError(f"StyleGAN: a hook on '{name}' is not supported: the fused synthesis chain has no stop "
                                          "point there (supported: blocks, epi1/epi2, style_mod(.lin), conv/conv0_up/conv1, "
                                          "torgb, g_synthesis)")
            act = self._run(w_layers, point)
            if m(_result=act) is not act:
                raise NotImplementedError(f"an edit on '{name}' cannot be propagated through the fused synthesis chain")

    def _block_modules(self, upto):
        for i, (name, blk) in enumerate(self.model.g_synthesis.blocks.items()):
            if i > upto:
                break
            pre = f"g_synthesis.blocks.{name}"
            for n, m in blk.named_modules(remove_duplicate=False):
                yield (f"{pre}.{n}" if n else pre), m

    def forward(self, x):
        """wrappers.py:368-370: 0.5 * (torgb(G_synthesis(w)) + 1) for one latent or a list of 18.  Hooked stop points of the
        synthesis network receive their activations."""
        w_layers = self._latents(x)
        n_blocks = len(self.model.g_synthesis.blocks)
        G = self.model.g_synthesis
        self._fire_hooks(w_layers, list(self._block_modules(n_blocks - 1)) + [("g_synthesis.torgb", G.torgb), ("g_synthesis", G)])
        out = self._run(w_layers, self._stop_points["g_synthesis"])
        return 0.5 * (out + 1)

    def feature_layout(self, layer_name):
        """Native (device) feature order of ``activations_into``: ('nhwc', (H, W, C)) for block / epilogue / conv outputs."""
        point = self._stop_points.get(layer_name)
        if point is None or point[1] not in ("epi", "conv"):
            return None
        res, co = self._synthesis().shapes[point[0]]
        return ("nhwc", (res, res, co))

    def activations_into(self, x, layer_name, out):
        """Activations of ``layer_name`` for latents x [n, 512] (in the current primary space) as fp32 NHWC rows written into
        ``out`` [n, H*W*C] (may be row-strided): the decomposition driver's producer for synthesis layers."""
        j, stop = self._stop_points[layer_name]
        w = x if self.w_primary else self.model.g_mapping(x)
        return self._synthesis().forward(w.reshape(1, -1, 512), j + 1, stop, out=out)

    def partial_forward(self, x, layer_name):
        """wrappers.py:373-417: map Z to W through the ``g_mapping`` module (its hooks fire), stop there for any ``g_mapping*``
        layer; otherwise run the synthesis blocks up to the first one with a child whose name contains ``layer_name`` (a
        substring match, as the reference), firing the hooks of that block and the ones before it.  No block -> the
        reference's RuntimeError."""
        w_layers = self._latents(x)
        if "g_mapping" in layer_name or layer_name == "truncation":
            return
        for i, (name, block) in enumerate(self.model.g_synthesis.blocks.items()):
            prefix = f"g_synthesis.blocks.{name}"
            leaves = [f"{prefix}.{n}" if n else prefix for n, m in block.named_modules(remove_duplicate=False) if not m._modules]
            if any(layer_name in c for c in leaves):
                self._fire_hooks(w_layers, list(self._block_modules(i)))
                return
        raise RuntimeError(f"Layer {layer_name} not encountered in partial_forward")

    def set_noise_seed(self, seed):
        """wrappers.py:420-436: every NoiseLayer gets randn(1, 1, H, W) drawn right after torch.random.manual_seed(seed)
        (so maps of one resolution are equal), in the reference's visiting order; drawn on the host."""
        def visit(m, name):
            for child_name, child in m._modules.items():
                if child is not None:
                    visit(child, f"{name}.{child_name}")
            if isinstance(m, stylegan.NoiseLayer):
                H, W = [int(v) for v in name.split(".")[2].split("x")]
                torch.random.manual_seed(seed)
                m.noise = torch.randn(1, 1, H, W, dtype=torch.float32).to(self.device)
        visit(self.model.g_synthesis, "g_synthesis")
        # (new maps may reuse the freed ones' addresses: the pack key counts the re-seeds)
        self._noise_generation = getattr(self, "_noise_generation", 0) + 1


# ---- factories (wrappers.py:651-735) ---------------------------------------------------------------
@singledispatch
def get_model(name, output_class, device, **kwargs):
    inst = kwargs.get("inst", None)
    model = kwargs.get("model", None)
    if inst or model:
        cached = model or inst.model
        network_same = cached.model_name == name
        outclass_same = cached.outclass == output_class
        can_change_class = "BigGAN" in name
        if network_same and (outclass_same or can_change_class):
            cached.set_output_class(output_class)
            return cached
    if name == "StyleGAN2":
        model = StyleGAN2(device, class_name=output_class, random_init=kwargs.get("random_init"))
    elif "BigGAN" in name:
        assert "-" in name, "Please specify BigGAN resolution, e.g. BigGAN-512"
        from .biggan import BigGAN
        model = BigGAN(device, name.split("-")[-1], class_name=output_class, random_init=kwargs.get("random_init"))
    elif name == "StyleGAN":
        model = StyleGAN(device, class_name=output_class, random_init=kwargs.get("random_init"))
    elif name in ("ProGAN", "DCGAN"):
        raise RuntimeError(f"{name} is outside the B200 hot path (SURVEY.md section 2: not in any BASELINE config)")
    else:
        raise RuntimeError(f"Unknown model {name}")
    return model


@get_model.register(Config)
def _(cfg, device, **kwargs):
    kwargs["use_w"] = kwargs.get("use_w", cfg.use_w)
    return get_model(cfg.model, cfg.output_class, device, **kwargs)


def _annotate_shapes(inst, model, layers):
    """The reference runs one full forward on zeros to record shapes (modelconfig.py:110-144).  Only the
    hooked layers' shapes and the latent shape are consumed by GANSpace, so a partial forward suffices."""
    input_shape = model.get_latent_shape()
    inst.retain_layers(layers)
    with torch.no_grad():
        dry = torch.zeros(input_shape, device=model.device)
        for layer in layers:
            model.partial_forward(dry, layer)
    inst.input_shape = input_shape
    inst.feature_shape = {layer: feat.shape for layer, feat in inst.retained_features().items()}
    inst.output_shape = None   # full image synthesis: SURVEY.md section 8(f) item 2
    return inst


@singledispatch
def get_instrumented_model(name, output_class, layers, device, **kwargs):
    model = get_model(name, output_class, device, **kwargs)
    model.eval()
    inst = kwargs.get("inst", None)
    if inst:
        inst.close()
    if not isinstance(layers, list):
        layers = [layers]
    module_names = [n for (n, _) in model.named_modules()]
    for layer_name in layers:
        if layer_name not in module_names:
            print(f"Layer '{layer_name}' not found in model!")
            print("Available layers:", "\n".join(module_names))
            raise RuntimeError(f"Unknown layer '{layer_name}''")
    if hasattr(model, "use_z"):
        model.use_z()
    inst = _annotate_shapes(InstrumentedModel(model), model, layers)
    if kwargs.get("use_w", False):
        model.use_w()
    return inst


@get_instrumented_model.register(Config)
def _(cfg, device, **kwargs):
    kwargs["use_w"] = kwargs.get("use_w", cfg.use_w)
    return get_instrumented_model(cfg.model, cfg.output_class, cfg.layer, device, **kwargs)
