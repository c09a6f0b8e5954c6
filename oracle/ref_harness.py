"""ORACLE / TEST INFRASTRUCTURE -- running the UNMODIFIED reference (harskish/ganspace) on the host CPU.

Only tests/, __graft_entry__ and bench.py's reference / cpu_baseline legs may import this module; nothing under
ganspace_b200/ does.

The reference is pure Python on this path (decomposition.get_or_compute -> models.wrappers.StyleGAN2 ->
stylegan2-pytorch Generator -> estimators.IPCAEstimator -> scikit-learn IncrementalPCA), so there is nothing to
compile: "installing" it means placing its *.py tree where the GPU box can import it.  ``install_ref()`` mirrors the
*.py files of /root/reference (1.3 MB; no checkpoints, images or notebooks) into baseline/_ref/, which is git-ignored
(never part of the repo's history) but NOT gpurun-ignored, so it travels to the B200 box like the built .so files.
``__graft_entry__.build()`` calls it whenever /root/reference is present.

``import_reference()`` is the recipe of SURVEY.md Appendix A: four sys.modules stubs for absent, non-hot-path imports
(fbpca, skimage, boto3, botocore) -- nothing of the reference itself is modified -- and ``RandInit*`` subclasses that
override only ``load_model`` (random-init weights under a fixed seed: there is no network for checkpoints and
BASELINE.json's configs say "random-init weights").
"""
import os
import shutil
import sys
import time
import types
from pathlib import Path
from types import SimpleNamespace

REPO = Path(__file__).resolve().parents[1]
REF_SRC = Path(os.environ.get("GANSPACE_REFERENCE", "/root/reference"))
REF_DST = REPO / "baseline" / "_ref"


def _is_file(p: Path) -> bool:
    """Path.is_file() that answers False, rather than raising, for a path the user may not read."""
    try:
        return p.is_file() and os.access(p, os.R_OK)
    except OSError:
        return False


def install_ref(src: Path = REF_SRC, dst: Path = REF_DST) -> bool:
    """Mirror the reference's *.py tree into baseline/_ref (idempotent).  False when the source is absent or unreadable."""
    src = Path(src)
    if not _is_file(src / "decomposition.py"):
        return False
    n = 0
    for p in src.rglob("*.py"):
        rel = p.relative_to(src)
        if rel.parts and rel.parts[0] in ("notebooks", "deps", "cache", "out"):
            continue
        q = dst / rel
        q.parent.mkdir(parents=True, exist_ok=True)
        if not q.exists() or q.stat().st_size != p.stat().st_size or q.read_bytes() != p.read_bytes():
            shutil.copyfile(p, q)
        n += 1
    (dst / "INSTALLED_FROM").write_text(f"{src} ({n} .py files, unmodified)\n")
    return True


def ref_dir():
    """Directory of an importable reference tree: /root/reference here, baseline/_ref on the GPU box; None if neither."""
    for d in (REF_SRC, REF_DST):
        if _is_file(d / "decomposition.py") and _is_file(d / "models" / "wrappers.py"):
            return d
    return None


_imported = None


def import_reference(ref=None):
    """-> namespace(wrappers, stylegan2, Config, decomposition, estimators, dir).  Imports the reference's top-level
    modules (config, decomposition, estimators, models, netdissect) under their own names -- do not mix with
    ganspace_b200's same-named modules in one interpreter unless they are imported as ``ganspace_b200.*``."""
    global _imported
    if _imported is not None:
        return _imported
    ref = Path(ref) if ref is not None else ref_dir()
    if ref is None:
        raise RuntimeError("no reference tree: neither /root/reference nor baseline/_ref exists (run __graft_entry__.build() "
                           "in the build container)")
    sys.path.insert(0, str(ref))

    def stub(name, **a):
        m = types.ModuleType(name)
        m.__dict__.update(a)
        sys.modules[name] = m
        return m

    for name in ("fbpca", "boto3"):
        if name not in sys.modules:
            stub(name)
    if "skimage" not in sys.modules:
        sk = stub("skimage")
        sk.morphology = stub("skimage.morphology")
    if "botocore" not in sys.modules:
        bc = stub("botocore")
        bc.exceptions = stub("botocore.exceptions", ClientError=Exception)
    cwd = os.getcwd()
    from models import wrappers, stylegan2          # noqa: chdir side effect (models/stylegan2/__init__.py:8-16)
    from config import Config
    import decomposition
    import estimators
    os.chdir(cwd)
    _imported = SimpleNamespace(wrappers=wrappers, stylegan2=stylegan2, Config=Config, decomposition=decomposition,
                                estimators=estimators, dir=ref)
    return _imported


def rand_init_stylegan2(ref, device, outclass="ffhq", seed=1234):
    """The reference's StyleGAN2 wrapper with random-init weights (load_model is the only override)."""
    import torch

    class RandInitStyleGAN2(ref.wrappers.StyleGAN2):
        def load_model(self):                      # replaces the checkpoint download (wrappers.py:153-165)
            torch.manual_seed(seed)
            self.model = ref.stylegan2.Generator(self.resolution, 512, 8).to(self.device)
            self.latent_avg = torch.zeros(512, device=self.device)

    return RandInitStyleGAN2(device, outclass)


def run_reference_style(n, b, c, use_w=True, outclass="ffhq", model=None, quiet=True, keep=False):
    """One unmodified ``decomposition.get_or_compute(force_recompute=True)`` of the reference on the CPU for
    layer=style; returns (seconds of the call, arrays or None).  Model construction is outside the timed span, as in
    the reference's own "Total time" print (decomposition.py:398-400)."""
    import tempfile
    import numpy as np
    import torch
    ref = import_reference()
    dev = torch.device("cpu")
    m = model if model is not None else rand_init_stylegan2(ref, dev, outclass)
    inst = ref.wrappers.get_instrumented_model("StyleGAN2", outclass, "style", dev, model=m, use_w=use_w)
    cfg = ref.Config(model="StyleGAN2", layer="style", output_class=outclass, estimator="ipca", use_w=use_w,
                     n=n, batch_size=b, components=c)
    out = None
    with tempfile.TemporaryDirectory() as tmp:
        old = sys.stdout, sys.stderr
        devnull = open(os.devnull, "w")
        if quiet:
            sys.stdout = sys.stderr = devnull
        try:
            t0 = time.perf_counter()
            path = ref.decomposition.get_or_compute(cfg, inst, force_recompute=True,
                                                    submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp))
            dt = time.perf_counter() - t0
        finally:
            sys.stdout, sys.stderr = old
            devnull.close()
        if keep:
            with np.load(path) as data:
                out = {k: data[k].copy() for k in data.files}
    return dt, out


DEEP512 = [(False, 16, 16), (True, 16, 16), (False, 16, 16), (True, 16, 8), (False, 8, 8), (True, 8, 8), (False, 8, 8),
           (True, 8, 4), (False, 4, 4), (True, 4, 2), (False, 2, 2), (True, 2, 1), (False, 1, 1), (True, 1, 1)]


def rand_init_biggan512(ref, device, outclass="husky", seed=4321):
    """The reference's BigGAN wrapper, biggan-deep-512 configuration, random init; 'husky' -> ImageNet class 248 (WordNet is
    absent here, so one_hot_from_names is replaced by its result for this one name; SURVEY.md Appendix A)."""
    import torch
    from models import biggan
    import models.wrappers as mw
    one_hot = lambda names: biggan.one_hot_from_int([248])
    biggan.one_hot_from_names = one_hot
    mw.biggan.one_hot_from_names = one_hot

    class RandInitBigGAN(ref.wrappers.BigGAN):
        def load_model(self, name):
            torch.manual_seed(seed)
            cfg = biggan.BigGANConfig(output_dim=512, layers=DEEP512, attention_layer_position=8)
            self.model = biggan.BigGAN(cfg).to(self.device)

    return RandInitBigGAN(device, 512, outclass)


def run_reference_config(w, n, keep=False, quiet=True):
    """One unmodified reference get_or_compute(force_recompute=True) for a bench.py WORKLOADS entry ``w`` at ``n`` samples;
    returns seconds (or (seconds, arrays) with keep=True).  Model construction is outside the timed span."""
    import tempfile
    import numpy as np
    import torch
    ref = import_reference()
    dev = torch.device("cpu")
    if w["model"].startswith("BigGAN"):
        m = rand_init_biggan512(ref, dev, w["output_class"], w["seed"])
        inst = ref.wrappers.get_instrumented_model(w["model"], w["output_class"], w["layer"], dev, model=m)
    else:
        m = rand_init_stylegan2(ref, dev, w["output_class"], w["seed"])
        inst = ref.wrappers.get_instrumented_model("StyleGAN2", w["output_class"], w["layer"], dev, model=m, use_w=w["use_w"])
    cfg = ref.Config(model=w["model"], layer=w["layer"], output_class=w["output_class"], estimator="ipca", use_w=w["use_w"],
                     n=n, batch_size=w["batch_size"], components=w["components"])
    out = None
    with tempfile.TemporaryDirectory() as tmp:
        old = sys.stdout, sys.stderr
        devnull = open(os.devnull, "w")
        if quiet:
            sys.stdout = sys.stderr = devnull
        try:
            t0 = time.perf_counter()
            path = ref.decomposition.get_or_compute(cfg, inst, force_recompute=True,
                                                    submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp))
            dt = time.perf_counter() - t0
        finally:
            sys.stdout, sys.stderr = old
            devnull.close()
        if keep:
            with np.load(path) as data:
                out = {k: data[k].copy() for k in data.files}
    inst.close()
    return (dt, out) if keep else dt


class limit_threads:
    """Context: cap torch's intra-op threads and the BLAS/OpenMP pools NumPy/SciPy use to ``t`` (None = leave as is)."""

    def __init__(self, t):
        self.t = t

    def __enter__(self):
        if self.t is None:
            return self
        import torch
        from threadpoolctl import threadpool_limits
        self.old = torch.get_num_threads()
        torch.set_num_threads(int(self.t))
        self.ctl = threadpool_limits(limits=int(self.t))
        return self

    def __exit__(self, *a):
        if self.t is None:
            return
        import torch
        self.ctl.restore_original_limits()
        torch.set_num_threads(self.old)


if __name__ == "__main__":
    print("installed:", install_ref(), "->", REF_DST)
