"""bench.py -- latent samples/sec into PCA (BASELINE.json metric) on N B200s.

Default workload = BASELINE.json configs[1] ("config 2"): StyleGAN2-ffhq (random-init weights, torch.manual_seed(1234)),
layer=style --use_w, N=1_000_000 b=10_000 c=80, estimator=ipca.  ``--config {1,3,4,5}`` selects the other BASELINE
configurations (same JSON line, same timing rules).  One "step" = one whole get_or_compute(force_recompute=True) over the N
samples (synthetic data: the latents ARE the data).

  value     N / device time of decomposition.compute_arrays() (CUDA events; seeds/weights resident; no file)
  e2e       N / wall time of the public get_or_compute() call: host seeds -> H2D, components D2H, .npz written
  roofline  the dominant producer kernel of the config (config 1-3: the fused mapping-network kernel, 4,194,304 FLOP per
            latent = 8 x 2*512*512, SURVEY.md section 8d), timed live with CUDA events around every launch inside the timed
            steps, against the measured bf16 peak in MEASURED_PEAKS.json.  ``frac`` = that kernel alone; ``frac_e2e`` =
            section 8d's whole-job definition (value x FLOP/sample / peak).  ``traffic`` comes from the committed ncu capture
            named in ``traffic_source`` (profiles/roofline_traffic.json), null when there is none for the kernel.
  parity    size-independent properties of the timed result + a small-N run of the same config compared with the oracle
  cpu_baseline  the reference arm on a bounded sample, run as a subprocess (CPU only) after the timed region

--dump-outputs DIR writes the arrays of the last timed step as DIR/<name>.npy; the inputs are seeded, so two builds run with the
same arguments can be compared output for output.

--impl reference times the UNMODIFIED reference (baseline/_ref = the *.py tree of harskish/ganspace, installed by
__graft_entry__.build(); oracle/ref_harness.py) through its own decomposition.get_or_compute on the host cores, one bounded
sample of the workload per step (default N=100_000 of the 1e6: the path's cost is linear in the number of 10k batches).  The
warm-up steps double as a thread-count sweep (torch intra-op + BLAS pools) and the timed steps use the fastest setting; one
extra full-size run (N=1e6) is appended when --ref-full is given or the time budget allows.  If baseline/_ref is absent the
arm falls back to the oracle port (kind "port").  Multi-GPU: launched by torchrun, one rank per GPU, NCCL; the job's N is
fixed (strong scaling of the one PCA job).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path
from types import SimpleNamespace

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# BASELINE.json configs (SURVEY.md section 8d).  flop = algorithmic FLOP per sample of the config's producer network.
WORKLOADS = {
    1: dict(model="StyleGAN2", output_class="ffhq", layer="style", use_w=True, n=10_000, batch_size=1_000, components=32,
            seed=1234, flop=8 * 2 * 512 * 512, section="mapping", small=dict(n=4_000, batch_size=1_000, components=32),
            name="StyleGAN2 random-init mapping net, layer=style --use_w (BASELINE.json configs[0])"),
    2: dict(model="StyleGAN2", output_class="ffhq", layer="style", use_w=True, n=1_000_000, batch_size=10_000, components=80,
            seed=1234, flop=8 * 2 * 512 * 512, section="mapping", small=dict(n=40_000, batch_size=10_000, components=80),
            name="StyleGAN2-ffhq random-init W-space PCA (layer=style --use_w) (BASELINE.json configs[1])"),
    3: dict(model="StyleGAN2", output_class="car", layer="style", use_w=False, n=1_000_000, batch_size=10_000, components=80,
            seed=1234, flop=8 * 2 * 512 * 512, section="mapping", small=dict(n=30_000, batch_size=10_000, components=80),
            name="StyleGAN2-car random-init Z-space layer=style PCA + latent regression (BASELINE.json configs[2])"),
    4: dict(model="BigGAN-512", output_class="husky", layer="generator.gen_z", use_w=False, n=1_000_000, batch_size=2_000,
            components=80, seed=4321, flop=2 * 256 * 32768, section="linear", small=None,
            name="BigGAN-512 husky random-init layer=generator.gen_z PCA + latent regression (BASELINE.json configs[3])"),
    5: dict(model="StyleGAN2", output_class="ffhq", layer="convs.4", use_w=False, n=200_000, batch_size=2_000, components=80,
            seed=1234, flop=3.17e9, section="synthesis", small=None,
            name="StyleGAN2-ffhq random-init conv feature map layer=convs.4 (d=524288) PCA + latent regression "
                 "(BASELINE.json configs[4]; g_synthesis.blocks.4 does not exist for StyleGAN2, SURVEY.md section 0.5)"),
}
METRICS = {
    1: "latent samples/sec into PCA (StyleGAN2 W, N=1e4)",
    2: "latent samples/sec into PCA (StyleGAN2-ffhq W, N=1e6)",
    3: "latent samples/sec into PCA (StyleGAN2-car Z layer=style, N=1e6)",
    4: "latent samples/sec into PCA (BigGAN-512 gen_z, N=1e6)",
    5: "latent samples/sec into PCA (StyleGAN2-ffhq convs.4, N=2e5)",
}


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def _workload(args):
    w = dict(WORKLOADS[args.config])
    for k, a in (("n", args.n), ("batch_size", args.batch), ("components", args.components)):
        if a is not None:
            w[k] = a
    return w


def _config_dict(w, world):
    if world > 1:
        par = ("feature-sharded chain over %d ranks (row-parallel synthesis, all-to-all, Gram all-reduce)" % world
               if w["layer"].startswith("convs") else
               "partial_fit groups k mod %d per rank; per-group (mean, Gram) statistics all-gathered as produced; "
               "merge chain replayed on every rank" % world)
    else:
        par = "single GPU"
    return {"workload": f"{w['name']}, N={w['n']} b={w['batch_size']} c={w['components']}, estimator=ipca",
            "parallelism": par,
            "l2": "inputs larger than L2 (every step regenerates and streams its latents / activations), no flush needed"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc, self.lines, self.gpu = None, [], gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower() == "active":
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# reference arm (CPU only)
# ----------------------------------------------------------------------------------------------------------------------
def _ref_step(w, n_sample, threads):
    """One bounded-sample step of the reference arm -> (seconds, kind)."""
    from oracle import ref_harness as rh
    # always an explicit thread count: torchrun exports OMP_NUM_THREADS=1 to its workers, which would leave the "all cores"
    # setting of the sweep single-threaded
    threads = threads or (os.cpu_count() or 1)
    if rh.ref_dir() is not None:
        with rh.limit_threads(threads):
            dt = rh.run_reference_config(w, n_sample)
        return dt, "reference"
    # no reference tree on this box: the oracle's restatement of the same path (layer=style configs only)
    from oracle import ganspace_oracle as orc
    if w["layer"] != "style":
        raise RuntimeError("reference arm: baseline/_ref is missing and the oracle port covers layer=style only")
    ws, bs = orc.mapping_random_init(w["seed"])
    with rh.limit_threads(threads):
        t0 = time.perf_counter()
        orc.compute_stylegan2_style(ws, bs, n_sample, w["batch_size"], w["components"], w["use_w"], ipca="svd")
        dt = time.perf_counter() - t0
    return dt, "port"


class _StdoutToStderr:
    """fd-level: whatever the wrapped code (or a library under it) prints to stdout goes to stderr, so that stdout carries
    the one JSON line only (the reference's model.py prints at import)."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    with _StdoutToStderr():
        line = _reference_line(args)
    print(line)


def _reference_line(args):
    w = _workload(args)
    n_sample = min(args.ref_sample or {1: 10_000, 2: 100_000, 3: 50_000, 4: 4_000, 5: 4_000}[args.config], w["n"])
    n_sample = max(n_sample // w["batch_size"], 1) * w["batch_size"]
    cores = os.cpu_count() or 1
    # thread-count sweep during the warm-up steps; the timed steps use the fastest setting
    # (order: the settings that won on the 128-core GPU boxes first -- 16 threads ran this path 2-3x faster than all cores --
    # so that a short warm-up still finds the reference's best)
    cands = [t for t in (16, 32) if t < cores] + [None] + [t for t in (64, 8) if t < cores]
    if args.ref_threads:
        cands = [args.ref_threads]
    sweep, best = {}, cands[0]
    for i in range(args.warmup):
        t = cands[i % len(cands)]
        dt, kind = _ref_step(w, n_sample, t)
        key = str(t or cores)
        sweep[key] = min(sweep.get(key, 1e30), dt)
    if sweep:
        best_key = min(sweep, key=sweep.get)
        best = None if int(best_key) == cores and not args.ref_threads else int(best_key)
    times = []
    for _ in range(args.steps):
        dt, kind = _ref_step(w, n_sample, best)
        times.append(dt)
    dt = sum(times) / len(times)
    value = n_sample / dt
    used = best or cores
    full = None
    est_full = dt * w["n"] / n_sample
    if args.ref_full or (args.ref_full is None and n_sample < w["n"] and est_full < 240.0):
        dtf, _ = _ref_step(w, w["n"], best)
        full = {"n": w["n"], "seconds": dtf, "value": w["n"] / dtf, "threads": used}
    sample = (f"N={n_sample} of the config's N={w['n']} per step (same b={w['batch_size']}, c={w['components']}): "
              + ("the unmodified reference (baseline/_ref) through its own decomposition.get_or_compute on the CPU"
                 if kind == "reference" else "oracle port (no reference tree on this box)")
              + f"; {used} threads (fastest of the warm-up sweep {{threads: s}} = { {k: round(v, 2) for k, v in sweep.items()} })")
    return json.dumps({
        "impl": "reference", "metric": METRICS[args.config], "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config_dict(w, args.gpus),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": used, "host_cores": cores, "kind": kind, "sample": sample,
                         "thread_sweep_s": sweep, "full_n": full},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def _cpu_baseline_subprocess(args):
    """The reference arm on one bounded sample, in a CPU-only subprocess (the reference picks 'cuda' when it sees one)."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--config", str(args.config), "--steps", "1",
           "--warmup", "2", "--no-ref-full"]
    if args.ref_sample:
        cmd += ["--ref-sample", str(args.ref_sample)]
    for k, a in (("--n", args.n), ("--batch", args.batch), ("--components", args.components)):
        if a is not None:
            cmd += [k, str(a)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        return json.loads(line)["cpu_baseline"]
    except Exception as e:                                   # the baseline is a reported extra, never fatal to the bench line
        return {"value": None, "unit": "samples/s", "cores": None, "kind": "unavailable", "sample": f"{type(e).__name__}: {e}"}


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def _props(out):
    import numpy as np
    c = out["act_comp"].shape[0]
    comp = out["act_comp"].reshape(c, -1).astype(np.float64)
    lat = out["lat_comp"].reshape(c, -1).astype(np.float64)
    return {"act_comp_orthonormality_err": float(np.max(np.abs(comp @ comp.T - np.eye(c)))),
            "lat_rows_unit_norm_err": float(np.max(np.abs(np.linalg.norm(lat, axis=1) - 1))),
            "var_ratio_sum": float(out["var_ratio"].sum()),
            "act_stdev_sorted": bool(np.all(np.diff(out["act_stdev"]) <= 0)),
            "finite": bool(all(np.isfinite(v).all() for v in out.values()))}


DUMP_BYTES = 64 << 20


def _dump_outputs(arrays, out_dir):
    """--dump-outputs: the float32 arrays compute_arrays() returned, as <out_dir>/<name>.npy, so that two builds can be compared
    output for output.  Each array gets an equal share of DUMP_BYTES; a larger one (act_comp of a conv layer: 168 MB at convs.4)
    is replaced by a sample of its flattened elements at positions drawn from a fixed seed, the same positions on every run."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        if a.nbytes > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(out_dir / f"{name}.npy", a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from ganspace_b200 import _native
    from ganspace_b200.config import Config
    from ganspace_b200 import decomposition
    from ganspace_b200.models import get_instrumented_model, get_model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout at the first collective; keep stdout for the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    _native.load()

    w = _workload(args)
    model = get_model(w["model"], w["output_class"], dev, random_init=w["seed"])
    inst = get_instrumented_model(w["model"], w["output_class"], w["layer"], dev, model=model, use_w=w["use_w"])

    def cfg(**over):
        kw = dict(model=w["model"], layer=w["layer"], output_class=w["output_class"], components=w["components"], n=w["n"],
                  batch_size=w["batch_size"], use_w=w["use_w"], estimator="ipca")
        kw.update(over)
        return Config(**kw)

    tmp = tempfile.mkdtemp(prefix="gsb_bench_")
    sub = SimpleNamespace(run_dir=tmp, run_dir_root=tmp)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    devnull = open(os.devnull, "w")

    def quiet(fn):
        old = sys.stdout
        sys.stdout = devnull
        try:
            return fn()
        finally:
            sys.stdout = old

    # ---- warm-up (both entry points) ----------------------------------------------------------------
    for _ in range(args.warmup):
        quiet(lambda: decomposition.compute_arrays(cfg(), inst))
    quiet(lambda: decomposition.get_or_compute(cfg(), inst, submit_config=sub, force_recompute=True))

    # ---- timed: device pipeline (value) + live per-kernel sections (roofline) -------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _native.instrument.reset()
    _native.instrument.timing = True
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = quiet(lambda: decomposition.compute_arrays(cfg(), inst))
    e1.record()
    barrier()
    dev_ms = e0.elapsed_time(e1) / args.steps
    sections = _native.instrument.section_ms()
    launches = _native.instrument.launches
    rows = dict(_native.instrument.rows)
    _native.instrument.timing = False

    # ---- timed: end to end through the public API (host seeds in, .npz out) ---------------------------
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        path = quiet(lambda: decomposition.get_or_compute(cfg(), inst, submit_config=sub, force_recompute=True))
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    if args.dump_outputs and rank == 0:
        _dump_outputs(last, args.dump_outputs)

    # ---- the roofline kernel alone (outside the timed region): same rows, nothing else on the GPU -------------------------
    isolated = None
    if w["section"] == "mapping" and rank == 0:
        rows_iso = int(rows.get("mapping", 0) // max(1, args.steps)) or w["n"]
        packed = model.model.style.packed()
        zi = torch.randn((rows_iso, 512), device=dev, dtype=torch.float32)
        oi = torch.empty_like(zi)
        for _ in range(2):
            packed.forward(zi, out=oi)
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); packed.forward(zi, out=oi); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        iso_ms = sorted(ts)[1]
        isolated = {"rows": rows_iso, "ms": iso_ms, "achieved": rows_iso * w["flop"] / (iso_ms * 1e-3) / 1e12}
        del zi, oi
    if world > 1:
        dist.barrier()

    # ---- parity (outside the timed region): properties of the full-size result; a small-N run vs the oracle ---------
    parity = None
    if rank == 0:
        with np.load(path) as data:
            full = {k: data[k] for k in data.files}
        parity = {"properties_full_size": _props(full)}
    if w.get("small") and w["layer"] == "style" and not args.no_parity:
        small = quiet(lambda: decomposition.compute_arrays(cfg(**w["small"]), inst))      # collective: every rank runs it
        if rank == 0:
            from oracle import ganspace_oracle as orc
            ws, bs = orc.mapping_random_init(w["seed"])
            s = w["small"]
            ref = orc.compute_stylegan2_style(ws, bs, s["n"], s["batch_size"], s["components"], w["use_w"])
            cmp = orc.compare_npz(small, ref)
            parity["vs_oracle_small_n"] = {"n": s["n"], "b": s["batch_size"], "c": s["components"],
                                           **{k: float(v) for k, v in cmp.items()}}
            parity["ok"] = bool(cmp["min_signed_cos"] >= 0.999 and cmp["max_abs_dvar_ratio"] <= 1e-3
                                and parity["properties_full_size"]["finite"])

    if rank == 0:
        N = decomposition._plan.make_plan(w["n"], w["batch_size"], w["components"]).N
        peaks, peak_kind = _peaks()
        peak = peaks["bf16_tflops_sustained"]
        sec = w["section"]
        sec_ms, sec_calls = sections.get(sec, (0.0, 0))
        sec_rows = rows.get(sec, 0)                               # rows the section's kernels processed on THIS rank
        sec_ms_step = sec_ms / args.steps
        achieved = (sec_rows / args.steps) * w["flop"] / (sec_ms_step * 1e-3) / 1e12 if sec_ms_step > 0 and sec_rows else None
        if args.config == 4 and os.environ.get("GANSPACE_B200_BIGGAN_AFFINE", "1") != "0":
            achieved = None      # low-rank shortcut (DESIGN.md 5a): the [N, 32768] gen_z product is never formed, only its 128-dim factor
        value = N / (dev_ms * 1e-3)
        d2h = int(sum(v.nbytes for v in full.values()))
        pl = decomposition._plan.make_plan(w["n"], w["batch_size"], w["components"])
        traffic, traffic_src = None, None
        tp = ROOT / "profiles" / "roofline_traffic.json"
        if tp.exists():
            tj = json.loads(tp.read_text()).get(_native.kernel_name(sec))
            if tj:
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
        out = {
            "metric": METRICS[args.config], "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config_dict(w, world),
            "e2e": {"value": N / (e2e_ms * 1e-3), "unit": "samples/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": 4 * (pl.n_calls + 1), "d2h_bytes_per_step": d2h},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": _native.kernel_name(sec),
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None,
                         "frac_e2e": value * w["flop"] / 1e12 / peak / world,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "note": "achieved = algorithmic FLOP of the rows this rank pushed through the kernel / live CUDA-event "
                                 "time of its launches inside the timed steps (other streams share the GPU); frac_e2e = "
                                 "value x FLOP/sample / (peak x n_gpus), SURVEY.md section 8d",
                         "peak_source": f"bf16_tflops_sustained, {peak_kind} (MEASURED_PEAKS.json)",
                         "ms_per_step": sec_ms_step, "launches_per_step": sec_calls / max(1, args.steps),
                         "rows_per_step": sec_rows / max(1, args.steps),
                         "isolated": (dict(isolated, frac=isolated["achieved"] / peak, frac_of_burst_peak=isolated["achieved"] / peaks["bf16_tflops"],
                                           note="the same kernel on the same number of rows with nothing else running, measured "
                                                "after the timed region (median of 3)") if isolated else None)},
            "sections_ms_per_step": {k: v[0] / args.steps for k, v in sections.items()},
            # strong scaling of ONE job: the sequential merge chain (small-d: replicated on every rank; feature maps: its
            # small-side eigen-solve) does not shrink with the GPU count -- the residual Amdahl term of the scaling run
            "amdahl": {"term": "merge chain (sequential rank-c merges; replicated on every rank for d <= 1024, small-side "
                               "eigen-solve replicated for feature maps)",
                       "ms_per_step": (sections["chain"][0] / args.steps) if "chain" in sections else None,
                       "of_ms_per_step": dev_ms},
            "parity": parity,
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = _cpu_baseline_subprocess(args)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--n", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--components", type=int, default=None)
    ap.add_argument("--ref-sample", dest="ref_sample", type=int, default=None)
    ap.add_argument("--ref-threads", dest="ref_threads", type=int, default=None)
    ap.add_argument("--ref-full", dest="ref_full", action="store_true", default=None)
    ap.add_argument("--no-ref-full", dest="ref_full", action="store_false")
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-parity", dest="no_parity", action="store_true")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the arrays of the last step as DIR/<name>.npy (float32, at most 64 MB "
                         "in all; a larger array is replaced by a fixed, seeded sample of its elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""          # the reference picks 'cuda' when it sees one (decomposition.py:163-164)
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
