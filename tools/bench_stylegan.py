"""Timings of the StyleGAN (v1) path on one GPU (random-init weights, seed 1234), printed as JSON lines:

  * get_or_compute(Config(output_class='ffhq')) at the full default size (layer g_mapping, N = 300000, c = 80), Z and W space
  * forward() images/s at 1024^2, batch 1 and 8
  * one synthesis-block decomposition: g_synthesis.blocks.16x16 (d = 131072), N = 20000, B = 2000, c = 32
  * the reference on the host CPU (the mirrored tree under baseline/_ref) for g_mapping at N = 10000, with the linear
    extrapolation to N = 300000 (its per-sample work is constant: one batch of latents, one mapping pass, one IPCA step per batch)

Device times come from CUDA events around calls that end in a synchronise; the card's name and power limit are read in the
same run.  Usage: python tools/bench_stylegan.py [--no-reference] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path
from types import SimpleNamespace

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from ganspace_b200.config import Config  # noqa: E402
from ganspace_b200.decomposition import get_or_compute  # noqa: E402
from ganspace_b200.models import StyleGAN, get_instrumented_model  # noqa: E402

DEV = torch.device("cuda:0")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, reps):
    """Device milliseconds of each of ``reps`` calls (events on the current stream, synchronised after each)."""
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def decomposition(model, quiet=True, **kw):
    cfg = Config(output_class="ffhq", **kw)
    inst = get_instrumented_model(cfg, DEV, model=model)

    def run():
        with tempfile.TemporaryDirectory() as tmp:
            old = sys.stdout
            if quiet:
                sys.stdout = open(os.devnull, "w")
            try:
                get_or_compute(cfg, inst, submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp), force_recompute=True)
            finally:
                if quiet:
                    sys.stdout.close()
                    sys.stdout = old
    run()                                                  # warm-up: module load, packing, scratch buffers
    ms = timed(run, 3)
    inst.close()
    model.use_z()
    return ms


def reference_cpu(n=10_000, b=1_000, c=80):
    from oracle import ref_harness as rh
    from oracle.gen_golden_sg1 import rand_init_stylegan
    ref = rh.import_reference()
    m = rand_init_stylegan(ref, torch.device("cpu"), "ffhq")
    res = {}
    for use_w in (False, True):
        cfg = ref.Config(output_class="ffhq", n=n, batch_size=b, components=c, use_w=use_w)
        inst = ref.wrappers.get_instrumented_model(cfg, torch.device("cpu"), model=m)
        with tempfile.TemporaryDirectory() as tmp:
            old = sys.stdout, sys.stderr
            sys.stdout = sys.stderr = open(os.devnull, "w")
            try:
                t0 = time.perf_counter()
                ref.decomposition.get_or_compute(cfg, inst, force_recompute=True,
                                                 submit_config=SimpleNamespace(run_dir=tmp, run_dir_root=tmp))
                dt = time.perf_counter() - t0
            finally:
                sys.stdout.close()
                sys.stdout, sys.stderr = old
        inst.close()
        res["w" if use_w else "z"] = dt
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-reference", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [{"card": card(), "torch": torch.__version__}]
    model = StyleGAN(DEV, "ffhq", random_init=1234)
    for use_w in (False, True):
        ms = decomposition(model, n=300_000, components=80, use_w=use_w)
        lines.append({"what": f"get_or_compute g_mapping {'W' if use_w else 'Z'} N=300000 c=80 (B automatic)", "ms": ms,
                      "samples_per_s": 300_000 / (min(ms) / 1e3)})
    with torch.no_grad():
        for bsz in (1, 8):
            z = model.sample_latent(bsz, seed=5)
            model.forward(z)
            ms = timed(lambda: model.forward(z), 10)
            lines.append({"what": f"forward 1024^2 batch {bsz}", "ms": ms, "images_per_s": bsz / (min(ms) / 1e3)})
    ms = decomposition(model, layer="g_synthesis.blocks.16x16", n=20_000, batch_size=2_000, components=32)
    lines.append({"what": "get_or_compute g_synthesis.blocks.16x16 (d=131072) Z N=20000 B=2000 c=32", "ms": ms,
                  "samples_per_s": 20_000 / (min(ms) / 1e3)})
    if not args.no_reference:
        r = reference_cpu()
        for k, dt in r.items():
            lines.append({"what": f"reference CPU get_or_compute g_mapping {k.upper()} N=10000 c=80 B=1000", "s": dt,
                          "extrapolated_s_at_N300000": dt * 30, "cpu_threads": torch.get_num_threads()})
    text = "\n".join(json.dumps(l) for l in lines)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
