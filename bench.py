#!/usr/bin/env python
"""Benchmark of the DGMR GAN training step on the B200-native path.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torch.distributed.run)
    python bench.py --impl reference --steps K --warmup W    (reference arm: the UNMODIFIED reference on the host cores)
    python bench.py --config c2|c3|c5  --mode native|dropin  --precision tf32|3xtf32   (other BASELINE.json configs / modes)
    python bench.py ... --dump-outputs DIR   (also write what the last timed step computed as DIR/<name>.npy)

One "step" (default config c3, BASELINE.json configs[2]; configs[3] when N > 1) = one full GAN step: 2 discriminator updates + 1
generator update, hinge + grid-cell losses, Adam, on a synthetic batch of 16 4->18-frame 256x256 radar sequences per GPU (weak
scaling, NCCL all-reduce of the flat G/D gradient buffers).  Prints ONE JSON line on rank 0.

What the line carries besides the contract's keys:
  roofline             the dominant tcgen05 launch (largest share of the instrumented step), per launch, plus the aggregate over all
                       tensor-core launches (conv fwd/dgrad, tap-split, wgrad)
  cpu_baseline         the reference's own `DGMR.training_step` (baseline/_ref; oracle port if absent) on the host cores, bounded sample
  reference_gpu_eager  the reference's own GPU path on the same B200: unmodified modules `.cuda()`, PyTorch eager + cuDNN, the wrapper's
                       literal schedule as shipped (autograd anomaly mode on) and with anomaly mode off, and the minimal schedule the
                       native arm runs -- the denominators of the ">= 5x the cuDNN-backed step" target
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_G = 521.4e9   # forward FLOPs (2*MAC) of the generator per sample, paper config (SURVEY.md 8d)
F_D = 35.7e9    # forward FLOPs of both discriminators per 22-frame sequence
METRIC = "radar frames/sec (G+D step, 256x256, 4->18)"

# BASELINE.json configs (SURVEY.md 8d).  c3 is the headline (c4 = c3 per GPU under torchrun); c1 is the reference's CPU smoke case.
CONFIGS = {
    "c1": dict(size=128, forecast_steps=4, latent=384, context=192, batch=2, k=1, kind="step"),
    "c2": dict(size=256, forecast_steps=18, latent=768, context=384, batch=8, k=1, kind="inference"),
    "c3": dict(size=256, forecast_steps=18, latent=768, context=384, batch=16, k=1, kind="step"),
    "c5": dict(size=256, forecast_steps=18, latent=768, context=384, batch=16, k=6, kind="step"),
}


def flop_step(batch, k):
    """Parity-preserving minimal GAN-step FLOPs (SURVEY.md 8d): B*[2*(F_G + 6 F_D) + K*(3 F_G + 3 F_D)]."""
    return batch * (2 * (F_G + 6 * F_D) + k * (3 * F_G + 3 * F_D))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16=d.get("bf16_tflops", 1590.0), bf16_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


def workload_config(args, world):
    """The `config` object of the JSON line -- built the same way for both arms so that the driver can compare them."""
    c = CONFIGS[args.config]
    what = ("DGMR generator-only eval inference" if c["kind"] == "inference" else
            "DGMR full GAN step (G + spatial+temporal D, hinge + grid-cell, 2 D updates + 1 G update, Adam)")
    return dict(workload=f"{what}, 4->{c['forecast_steps']} frames 1x{c['size']}x{c['size']}, latent {c['latent']} / context {c['context']}, "
                         f"batch {args.batch}/GPU, generation_steps={args.generation_steps}",
                name=args.config + ("/c4" if (args.config == "c3" and world > 1) else ""),
                global_batch=world * args.batch, parallelism=f"dp{world}")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        smax = max([float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] + [0.0])
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=smax or None, reasons=sorted(reasons), samples=len(self.rows))


# ----------------------------------------------------------------------------------------------------- CPU arm
def build_oracle_state(cfg, seed=0):
    """Seeded construction through the package's parameter containers (CPU, no kernels)."""
    import skillful_nowcasting_b200 as B

    torch.manual_seed(seed)
    s = cfg["output_shape"]
    gen = B.Generator(B.ContextConditioningStack(input_channels=1, output_channels=cfg["context_channels"]),
                      B.LatentConditioningStack(shape=(8, s // 32, s // 32), output_channels=cfg["latent_channels"]),
                      B.Sampler(forecast_steps=cfg["forecast_steps"], latent_channels=cfg["latent_channels"],
                                context_channels=cfg["context_channels"]))
    disc = B.Discriminator(input_channels=1)
    return gen, disc


def usable_cores() -> int:
    """Host cores this process may really use: affinity mask and cgroup quota, not os.cpu_count() (on a box with a CPU quota,
    one thread per visible core oversubscribes the quota and torch crawls)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 32))     # the many small ops of this model do not scale past a few tens of threads


# bounded samples of the workload, largest first: (image side, forecast steps).  The discriminator needs side >= 128.
CPU_SAMPLES = ((128, 18), (128, 6), (128, 2))


def _cpu_child(argv):
    """Child process: time GAN steps of one bounded sample on the host cores, one JSON line per finished step (partial results
    survive a timeout).  kind 'reference': the UNMODIFIED reference's `DGMR.training_step` (literal schedule, anomaly mode off);
    kind 'port': the oracle port's minimal-schedule step."""
    kind = argv[0]
    side, t, batch, steps, k, lat, ctx, threads = (int(v) for v in argv[1:])
    torch.set_num_threads(threads)
    torch.manual_seed(1234)
    x, y = torch.rand(batch, 4, 1, side, side), torch.rand(batch, t, 1, side, side)
    cfg = dict(output_shape=side, forecast_steps=t, latent_channels=lat, context_channels=ctx)
    if kind == "reference":
        from baseline import reference_arm as R

        model = R.build_dgmr(cfg, generation_steps=k, anomaly=False)
        step = R.training_step_fn(model, x, y)
    else:
        from oracle import dgmr_oracle as O

        gen, disc = build_oracle_state(cfg)
        gs = O.clone_state(gen.state_dict(), requires_grad=True)
        ds = O.clone_state(disc.state_dict(), requires_grad=True)
        g_opt = O.AdamState([gs[n] for n in O._trainable(gs)], lr=5e-5)
        d_opt = O.AdamState([ds[n] for n in O._trainable(ds)], lr=2e-4)
        step = lambda: O.gan_step(gs, ds, g_opt, d_opt, x, y, t, (8, side // 32, side // 32), generation_steps=k)  # noqa: E731
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        print(json.dumps(dict(times=times)), flush=True)


def cpu_reference_steps(cfg, batch, steps, warmup, k, budget_s=150.0, samples=CPU_SAMPLES):
    """The reference's own CPU implementation of the path, timed on a BOUNDED sample of the workload and scaled to the metric's unit.

    What runs: the unmodified reference package (baseline/_ref, installed by `__graft_entry__.build()` where /root/reference exists)
    through its public `DGMR.training_step` -- kind "reference"; if that package is absent, the oracle port's step -- kind "port".
    A sample is the same step (same widths, same code) on smaller frames / fewer lead times / batch 1; its time is scaled by the
    pixel-and-frame ratio to the full-size step (convolution-dominated: cost ~ pixels x frames) and `value` = batch x frames / that.
    Exactly `warmup` untimed + `steps` timed steps run in a child process under a wall-clock budget; if the budget would be exceeded
    the next smaller sample is tried (a quota-limited host can be 10x slower than the build container)."""
    from baseline import reference_arm as R

    kind = "reference" if R.reference_root() else "port"
    threads = usable_cores()
    full_side, full_t = cfg["output_shape"], cfg["forecast_steps"]
    n_steps = max(1, steps + warmup)
    last_err = "no sample finished"
    for side, t in samples:
        side, t = min(side, full_side), min(t, full_t)
        cmd = [sys.executable, os.path.abspath(__file__), "--cpu-child", kind, str(side), str(t), str(batch), str(n_steps), str(k),
               str(cfg["latent_channels"]), str(cfg["context_channels"]), str(threads)]
        t_start = time.perf_counter()
        out = ""
        try:
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=budget_s, cwd=ROOT).stdout
        except subprocess.TimeoutExpired as e:
            out = e.stdout.decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
            last_err = f"sample {side}x{side} 4->{t} exceeded {budget_s:.0f} s"
        lines = [ln for ln in out.splitlines() if ln.startswith("{")]
        times = json.loads(lines[-1])["times"] if lines else []
        budget_s = max(30.0, budget_s - (time.perf_counter() - t_start))
        if len(times) == n_steps:
            timed = times[warmup:] if len(times) > warmup else times
            mean = sum(timed) / len(timed)
            scale = (full_side * full_side * full_t) / float(side * side * t)
            full_step_s = mean * scale
            what = ("UNMODIFIED reference package (dgmr 1.4.4, baseline/_ref): DGMR.training_step, its literal schedule, autograd anomaly mode off"
                    if kind == "reference" else "oracle port (oracle/dgmr_oracle.py), minimal schedule")
            return dict(value=batch * full_t / full_step_s, unit="frames/s", cores=threads, kind=kind, s_per_step=full_step_s,
                        steps_timed=len(timed), warmup_run=min(warmup, len(times) - len(timed)),
                        sample=f"{what}; same widths (latent {cfg['latent_channels']} / context {cfg['context_channels']}), generation_steps={k}, "
                               f"on {side}x{side} frames, 4->{t} lead times, batch {batch}: {len(timed)} timed step(s) of {mean:.2f} s after "
                               f"{len(times) - len(timed)} warm-up, " + (f"scaled x{scale:.1f} (pixels x frames) to the {full_side}x{full_side} 4->{full_t} step"
                                                                           if scale != 1.0 else "un-scaled (this IS the configuration)"))
        elif not out:
            last_err = last_err if "exceeded" in last_err else f"sample {side}x{side} 4->{t} produced no output"
    return dict(value=None, unit="frames/s", cores=threads, kind=kind, s_per_step=float("nan"), steps_timed=0, warmup_run=0,
                sample=f"unavailable: {last_err}")


def gpu_reference_eager(cfg, batch, k, dev):
    """The reference's own GPU path on this B200 (SURVEY.md 8d): the UNMODIFIED modules `.cuda()`, PyTorch eager + cuDNN with torch's
    defaults (cudnn.allow_tf32 = True).  Three measurements, each 1 warm-up + 2 timed steps with CUDA events:
      as_shipped        DGMR.training_step, autograd anomaly mode ON (the constructor switches it on globally, ref: dgmr/dgmr.py:130)
      anomaly_off       the same literal schedule with anomaly mode off
      minimal_schedule  the parity-preserving minimal schedule the native arm runs, on the reference's modules (apples to apples)
    A batch that does not fit is halved and the result says so."""
    from baseline import reference_arm as R

    if R.reference_root() is None:
        return dict(unavailable="reference package not found (baseline/_ref)")
    s, t = cfg["output_shape"], cfg["forecast_steps"]
    out = dict(what="unmodified reference modules on cuda:0, PyTorch eager + cuDNN (allow_tf32 default), fp32 storage", batch_requested=batch)

    def measure(fn_builder, b):
        torch.manual_seed(1234)
        x, y = torch.rand(b, 4, 1, s, s, device=dev), torch.rand(b, t, 1, s, s, device=dev)
        step = fn_builder(x, y)
        step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(2):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 2
        return dict(batch=b, ms_per_step=ms, value=b * t / (ms * 1e-3), unit="frames/s")

    for name, anomaly, minimal in (("anomaly_off", False, False), ("as_shipped", True, False), ("minimal_schedule", False, True)):
        b = batch
        while b >= 1:
            try:
                model = R.build_dgmr(cfg, generation_steps=k, anomaly=anomaly).to(dev)
                builder = (lambda x, y: R.minimal_step_fn(model, x, y)) if minimal else (lambda x, y: R.training_step_fn(model, x, y))
                out[name] = measure(builder, b)
                break
            except torch.cuda.OutOfMemoryError:
                out[name] = dict(batch=b, error="out of memory")
                b //= 2
            finally:
                model = None
                torch.cuda.empty_cache()
    torch.autograd.set_detect_anomaly(False)
    return out


# ----------------------------------------------------------------------------------------------------- GPU arm
_REAL_STDOUT = None


def emit(line: dict):
    """Write the ONE JSON line of the contract to the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_MAX_ELEMS = 8 << 20      # per output array (32 MB of fp32); a larger one is written as a fixed, seeded sample of this many elements
DUMP_PARAM_SAMPLE = 1 << 20   # elements sampled from each network's updated parameters


def _seeded_sample(t, k):
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:k].sort().values
    return t.reshape(-1)[idx.to(t.device)]


def dump_outputs(path, outputs, nets=None):
    """Write the arrays the last timed step returned (`outputs`: name -> tensor) as path/<name>.npy in float32, and for a training step
    `nets` = (generator, discriminator): a fixed, seeded sample of each network's parameters after that step's update, flattened in
    `.parameters()` order.  Arrays over DUMP_MAX_ELEMS elements are flattened and sampled the same way; at most ~40 MB in all."""
    import numpy as np

    arrays = {k: v.detach() for k, v in outputs.items()}
    for name, net in zip(("generator_params", "discriminator_params"), nets or ()):
        flat = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
        arrays[name] = _seeded_sample(flat, min(DUMP_PARAM_SAMPLE, flat.numel()))
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        if t.numel() > DUMP_MAX_ELEMS:
            t = _seeded_sample(t, DUMP_MAX_ELEMS)
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def main():
    # stdout must carry exactly one JSON line, but libraries print there too (NCCL's "NCCL version ..." banner under torchrun):
    # point fd 1 at stderr for the duration of the run and keep the real stdout for emit()
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS), help="BASELINE.json configuration (c3 = headline; c4 = c3 under torchrun)")
    ap.add_argument("--mode", default="native", choices=["native", "dropin"],
                    help="native: this repo's step driver (minimal schedule); dropin: the reference's unmodified dgmr/dgmr.py wrapper "
                         "(literal schedule, torch.optim.Adam) over this repo's modules (SURVEY.md 8d mode (i))")
    ap.add_argument("--precision", default="tf32", choices=["tf32", "3xtf32"], help="tensor-core operand mode: fast (1xTF32) or parity (3xTF32)")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the configuration's)")
    ap.add_argument("--generation-steps", type=int, default=None)
    ap.add_argument("--cuda-graph", action="store_true", help="c2 only: replay the eval forward from a CUDA graph (skillful_nowcasting_b200.inference)")
    ap.add_argument("--no-d-phase-graph", dest="d_phase_graph", action="store_false",
                    help="training configs: run the D phase's gradient-free generator forwards eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference's own GPU path (reference_gpu_eager)")
    ap.add_argument("--cpu-batch", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (and, for training, a fixed sample of the "
                         "updated parameters) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    c = CONFIGS[args.config]
    args.batch = args.batch or c["batch"]
    args.generation_steps = args.generation_steps or c["k"]
    cfg = dict(output_shape=c["size"], forecast_steps=c["forecast_steps"], latent_channels=c["latent"], context_channels=c["context"])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K = args.generation_steps
    config = workload_config(args, world)

    if args.impl == "reference":
        if rank != 0:
            return
        samples = ((c["size"], c["forecast_steps"]),) if args.config == "c1" else CPU_SAMPLES
        batch = c["batch"] if args.config == "c1" else args.cpu_batch
        r = cpu_reference_steps(cfg, batch, args.steps, args.warmup, K, budget_s=420.0, samples=samples)
        line = dict(impl="reference", metric=METRIC, value=r["value"], unit="frames/s", n_gpus=args.gpus,
                    steps=r["steps_timed"], warmup=r["warmup_run"], steps_requested=args.steps, warmup_requested=args.warmup,
                    ms_per_step=(r["s_per_step"] * 1e3 if r["value"] else None), higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32", data="synthetic", config=config,
                    cpu_baseline=dict(value=r["value"], unit="frames/s", cores=r["cores"], kind=r["kind"], sample=r["sample"]),
                    e2e=dict(value=r["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        emit(line)
        return

    import torch.distributed as dist
    from skillful_nowcasting_b200 import _lib, ops
    from skillful_nowcasting_b200.training import Adam, gan_step

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)
    be = _lib.backend()  # raises if libdgmr_b200.so is missing: no fallback
    ops.config.precision = 1 if args.precision == "3xtf32" else 0
    B, T, S = args.batch, c["forecast_steps"], c["size"]
    inference = c["kind"] == "inference"
    torch.manual_seed(1234 + rank)
    host_x = torch.rand(B, 4, 1, S, S).pin_memory()
    host_y = torch.rand(B, T, 1, S, S).pin_memory()
    x, y = host_x.to(dev), host_y.to(dev)
    host_out = torch.empty(B, T, 1, S, S).pin_memory() if c["kind"] == "inference" else None

    d_graph, d_graph_note = None, None
    if args.mode == "dropin":
        from baseline import reference_arm as R

        model = R.build_dgmr(cfg, generation_steps=K, dropin=True, anomaly=False, seed=0).to(dev)   # reference wrapper, our modules
        gen, disc = model.generator, model.discriminator

        def run_step(xi, yi):
            model.training_step((xi, yi), 0)
            lg = model.logged
            return {"d_loss": lg["train/d_loss"], "g_loss": lg["train/g_loss"], "grid_loss": lg["train/grid_loss"]}
    else:
        gen, disc = build_oracle_state(cfg, seed=0)  # identical replicas on every rank
        gen.to(dev)
        disc.to(dev)
        if inference:
            gen.eval()
            def run_eager(xi, yi):
                with torch.no_grad():
                    return {"out": gen(xi)}

            run_step = run_eager
            if args.cuda_graph:
                from skillful_nowcasting_b200.inference import GraphedGenerator

                runner = GraphedGenerator(gen, x)

                def run_step(xi, yi):
                    return {"out": runner(xi)}
        else:
            gen.train()
            disc.train()
            g_opt = Adam(gen.parameters(), lr=5e-5, betas=(0.0, 0.999))
            d_opt = Adam(disc.parameters(), lr=2e-4, betas=(0.0, 0.999))

            # the two gradient-free generator forwards of the D phase replay from a CUDA graph (launch-bound ConvGRU steps); the
            # instrumented step below runs them eagerly so that every launch carries its events
            d_graph_note = "eager"
            if args.d_phase_graph and args.precision == "tf32":
                try:
                    from skillful_nowcasting_b200.inference import GraphedGenerator

                    d_graph = GraphedGenerator(gen, x, train_mode=True)
                    d_graph_note = f"cuda-graph ({d_graph.launches} launches per replay)"
                except Exception as e:  # noqa: BLE001 -- a failed capture must not cost the measurement: run the eager path and say so
                    d_graph, d_graph_note = None, f"eager (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
                    print(f"bench: D-phase graph capture failed, running eagerly: {e}", file=sys.stderr)
                    torch.cuda.synchronize()

            def run_step(xi, yi, graphed=True):
                return gan_step(gen, disc, g_opt, d_opt, xi, yi, generation_steps=K, d_phase_generator=d_graph if graphed else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step_resident():
        last["out"] = run_step(x, y)
        return last["out"]

    def step_e2e():
        xi = host_x.to(dev, non_blocking=True)
        yi = host_y.to(dev, non_blocking=True)
        out = run_step(xi, yi)
        if inference:
            host_out.copy_(out["out"], non_blocking=True)     # device->host read of the forecast itself, into pinned memory
            torch.cuda.current_stream().synchronize()
            return host_out
        return torch.stack([out["d_loss"], out["g_loss"], out["grid_loss"]]).cpu()  # device->host read of the step's result

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = be.launches
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), be.launches - l0

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["out"], None if inference else (gen, disc))
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)

    # ---- roofline: one extra instrumented step, CUDA events (on the launch stream) around every C-ABI launch
    be.profile = []
    if inference and args.cuda_graph:
        run_eager(x, y)       # a graph replay issues no host launches: the per-launch events come from one eager forward of the same model
    elif not inference and args.mode != "dropin":
        run_step(x, y, graphed=False)
    else:
        step_resident()
    torch.cuda.synchronize()
    prof, be.profile = be.profile, None
    agg, shapes = {}, {}
    for name, flops, ev0, ev1, tag, info in prof:
        ms_ = ev0.elapsed_time(ev1)
        a = agg.setdefault(tag, [0.0, 0.0, 0])
        a[0] += flops; a[1] += ms_; a[2] += 1
        b_ = shapes.setdefault((tag, info), [0.0, 0.0, 0])
        b_[0] += flops; b_[1] += ms_; b_[2] += 1
    dump = os.environ.get("DGMR_BENCH_DUMP")
    if dump and rank == 0:
        with open(dump, "w") as f:
            f.write("tag\tshape\tcalls\tms\tTFLOP/s\n")
            for (tag, info), (fl, ms_, n_) in sorted(shapes.items(), key=lambda kv: -kv[1][1]):
                f.write(f"{tag}\t{info}\t{n_}\t{ms_:.3f}\t{(fl / (ms_ * 1e-3) / 1e12 if ms_ > 0 else 0):.1f}\n")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    ms_per_step = ms / args.steps
    frames = world * B * T
    value = frames / (ms_per_step * 1e-3)
    e2e_value = frames / (ms_e2e / args.steps * 1e-3)
    tf32_peak = pk["bf16_sustained"] / 2.0
    TC_TAGS = ("conv_umma", "conv_umma_splitk", "wgrad_umma")
    tc = [sum(agg.get(t, [0.0, 0.0, 0])[i] for t in TC_TAGS) for i in range(3)]
    instr_ms = sum(v[1] for v in agg.values())
    # the dominant launch = the (kernel family, shape) with the largest summed duration among the tensor-core launches
    top = max(((k_, v) for k_, v in shapes.items() if k_[0] in TC_TAGS), key=lambda kv: kv[1][1], default=(("none", ""), [0.0, 0.0, 1]))
    (top_tag, top_info), (top_fl, top_ms, top_n) = top
    top_ach = top_fl / (top_ms * 1e-3) / 1e12 if top_ms > 0 else 0.0
    agg_ach = tc[0] / (tc[1] * 1e-3) / 1e12 if tc[1] > 0 else 0.0
    if inference:
        h2d, d2h = int(host_x.numel()) * 4, int(B * T * S * S) * 4
        step_flops = world * B * F_G
    else:
        h2d, d2h = int(host_x.numel() + host_y.numel()) * 4, 12
        step_flops = flop_step(world * B, K)
    # DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the launches captured with `ncu --set full` and committed under
    # profiles/ (kernels_r02b_ncu.txt): reported for the dominant launch when it is one of them, else null
    NCU_TRAFFIC = {("conv_umma", "32x22x64x64 48->48 k333 G1"): (553955328 + 520765184, "profiles/kernels_r02b_ncu.txt (column-stacked CTA-pair kernel; algorithmic: 553.6 MB in + 553.6 MB out)"),
                   ("conv_umma", "288x1x64x64 96->96 k133 G18"): (908325120 + 424768256, "profiles/kernels_r02b_ncu.txt (CTA-pair halo-patch kernel; algorithmic: 453 MB in + 453 MB out + 453 MB residual)"),
                   ("wgrad_umma", "288x1x16x16 768->768 k133"): (739300352 + 15547904, "profiles/kernels_r02b_ncu.txt (row wgrad; algorithmic: 226 MB x + 226 MB dz, read once per filter row)")}
    top_traffic = NCU_TRAFFIC.get((top_tag, top_info.split(" (")[0].strip()))
    line = dict(
        metric=METRIC if not inference else "generated radar frames/sec (generator-only eval inference, 256x256, 4->18)",
        value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=warm, ms_per_step=ms_per_step, higher_is_better=True,
        scaling="weak", vs_baseline=None,
        dtype=("tf32 (fp32 storage, tcgen05 kind::tf32 operands, fp32 accumulate)" if args.precision == "tf32" else
               "3xtf32 (fp32 storage, error-compensated tf32 operand pairs on tcgen05, fp32 accumulate)"), data="synthetic",
        config=dict(config, mode=args.mode + ("+cuda-graph" if args.cuda_graph else ""), precision=args.precision,
                    l2="inputs+activations per step (>10 GB) exceed the 126 MB L2; no explicit flush needed",
                    schedule=("reference wrapper's literal schedule (checkpoint recompute, trailing forward), torch.optim.Adam" if args.mode == "dropin"
                              else "generator forward only, eval mode" if inference else "parity-preserving minimal schedule (SURVEY.md 8d)"),
                    **({"d_phase_generator_forwards": d_graph_note} if d_graph_note else {})),
        e2e=dict(value=e2e_value, unit="frames/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
        gpu_launches=launches // args.steps + (2 * d_graph.launches if d_graph is not None else 0),   # host launches + the kernels of the 2 graph replays
        clocks=clocks,
        step_tflops=step_flops / (ms_per_step * 1e-3) / 1e12,
        roofline=dict(bound="tensor", kernel=f"{top_tag} {top_info} (tcgen05 kind::tf32 implicit GEMM; the tensor-core launch with the largest share of the step)",
                      achieved=top_ach, peak=tf32_peak, unit="TFLOP/s", frac=top_ach / tf32_peak if tf32_peak else None,
                      traffic=(top_traffic[0] if top_traffic else None), traffic_source=(top_traffic[1] if top_traffic else None),
                      launches_per_step=top_n, ms_per_launch=top_ms / max(top_n, 1), share_of_step=top_ms / instr_ms if instr_ms else None,
                      peak_source=f"{pk['source']} bf16 sustained {pk['bf16_sustained']} TF/s / 2 (TF32 pipe = half the bf16 rate)",
                      note="achieved = executed FLOPs of one launch (2*pixels*Cin*Cout*taps) / its mean CUDA-event duration inside the instrumented step; "
                           "traffic (ncu dram bytes per launch) is recorded in profiles/ for the launches that were captured",
                      aggregate=dict(what="all tensor-core launches of the step: conv fwd + dgrad, tap-split, wgrad", achieved=agg_ach,
                                     frac=agg_ach / tf32_peak if tf32_peak else None, launches=tc[2], kernel_ms_per_step=tc[1],
                                     share_of_step=tc[1] / instr_ms if instr_ms else None)),
        kernel_breakdown_ms={k_: round(v[1], 3) for k_, v in sorted(agg.items(), key=lambda kv: -kv[1][1])},
    )
    # free the benchmark's own state before the reference's eager path needs the memory
    del prof
    if not args.no_ref_gpu and world == 1 and not inference and args.mode == "native":
        gen = disc = g_opt = d_opt = d_graph = None     # (the graph runner holds the generator and its private memory pool)
        ops.clear_pack_cache()
        gc.collect()
        torch.cuda.empty_cache()
        try:
            line["reference_gpu_eager"] = gpu_reference_eager(cfg, B, K, dev)
        except Exception as e:  # noqa: BLE001  (the headline number must survive a failure of the comparison arm)
            line["reference_gpu_eager"] = dict(error=f"{type(e).__name__}: {e}"[:400])
    if not args.no_cpu_baseline and world == 1:
        r = cpu_reference_steps(cfg, args.cpu_batch, 1, 0, K, budget_s=90.0)
        line["cpu_baseline"] = dict(value=r["value"], unit="frames/s", cores=r["cores"], kind=r["kind"], sample=r["sample"])
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--cpu-child":
        _cpu_child(sys.argv[2:])
    else:
        main()
