"""Time batched ensemble forecasts and the ensemble statistics kernel (measurement helper, not a test).

  python tests/time_ensemble.py OUT_DIR        ->  OUT_DIR/ensemble.json

Forward: C2 widths (latent 768, context 384), 256^2, 4 -> 18 frames, B = 8, eval mode, 1xTF32.  For each K the two arms are K replays of
the single-forecast CUDA graph (inference.GraphedGenerator(gen, x)) and one replay of the K-member graph (GraphedGenerator(gen, x,
num_samples=K)); they alternate, each timed with CUDA events over at least 1 s of work after two warm-up calls.
summarize: ensemble.summarize with a target and 3 thresholds on [8, K, 18, 1, 256, 256] (every input larger than the 126 MB L2), achieved
bandwidth of the algorithmic bytes 4 * P * B * (K + 1 target + 1 mean + 3 prob) against the 7.7 TB/s HBM3e data-sheet figure."""
import json
import math
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import skillful_nowcasting_b200 as B  # noqa: E402
from skillful_nowcasting_b200 import _lib  # noqa: E402
from skillful_nowcasting_b200.ensemble import summarize  # noqa: E402
from skillful_nowcasting_b200.inference import GraphedGenerator  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
BATCH, STEPS, SIZE = 8, 18, 256


def _events(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps          # ms per call


def time_forward(gen, x, single, K):
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    batched = GraphedGenerator(gen, x, num_samples=K)
    seq = lambda: [single(x) for _ in range(K)]
    one = lambda: batched(x)
    for f in (seq, one, seq, one):              # warm-up
        f()
    torch.cuda.synchronize()
    probe = _events(seq, 1) + _events(one, 1)
    reps = max(2, math.ceil(2.0 / (probe / 1e3)))   # >= 1 s per arm (probe: ms for one call of each arm)
    t_seq, t_one = [], []
    for _ in range(reps):                       # alternate the arms
        t_seq.append(_events(seq, 1))
        t_one.append(_events(one, 1))
    ms_seq, ms_one = sum(t_seq) / reps, sum(t_one) / reps
    frames = BATCH * K * STEPS
    M = gen.sampler.members_per_pass(BATCH, SIZE // 32, SIZE // 32)
    row = dict(K=K, reps=reps, sequential_ms=ms_seq, batched_ms=ms_one, speedup=ms_seq / ms_one,
               sequential_member_frames_per_s=frames / (ms_seq / 1e3), batched_member_frames_per_s=frames / (ms_one / 1e3),
               passes_per_call=math.ceil(K / M), members_per_pass=min(M, K), batched_graph_launches=batched.launches,
               sequential_graph_launches=K * single.launches, max_memory_allocated_GB=torch.cuda.max_memory_allocated() / 1e9,
               batched_graph_extra_memory_GB=(torch.cuda.memory_allocated() - base) / 1e9,
               sequential_ms_all=t_seq, batched_ms_all=t_one)
    del batched
    torch.cuda.empty_cache()
    return row


def time_summarize(K):
    g = torch.Generator(device="cuda").manual_seed(K)
    ens = torch.rand((BATCH, K, STEPS, 1, SIZE, SIZE), generator=g, device="cuda") * 10.0
    target = torch.rand((BATCH, STEPS, 1, SIZE, SIZE), generator=g, device="cuda") * 10.0
    thr = (0.5, 2.0, 8.0)
    f = lambda: summarize(ens, thr, target)
    for _ in range(3):
        f()
    torch.cuda.synchronize()
    reps = max(5, math.ceil(1.0 / (_events(f, 3) / 1e3)))
    ms = _events(f, reps)
    P = STEPS * SIZE * SIZE
    nbytes = 4.0 * P * BATCH * (K + 1 + 1 + len(thr))
    return dict(K=K, reps=reps, ms=ms, algorithmic_GB=nbytes / 1e9, GB_per_s=nbytes / (ms / 1e3) / 1e9,
                fraction_of_hbm_bound=nbytes / (ms / 1e3) / HBM_BYTES_PER_S)


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/time_ensemble.py OUT_DIR")
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    assert torch.cuda.is_available(), "time_ensemble.py needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    _lib.backend()
    torch.manual_seed(0)
    gen = B.Generator(B.ContextConditioningStack(input_channels=1, output_channels=384),
                      B.LatentConditioningStack(shape=(8, SIZE // 32, SIZE // 32), output_channels=768),
                      B.Sampler(forecast_steps=STEPS, latent_channels=768, context_channels=384)).cuda().eval()
    x = torch.rand((BATCH, 4, 1, SIZE, SIZE), device="cuda")
    t0 = time.time()
    single = GraphedGenerator(gen, x)
    res = dict(gpu=smi, config="C2 widths (latent 768, context 384), 256x256, 4->18 frames, B=8, eval, 1xTF32", forward=[], summarize=[])
    for K in (1, 4, 8, 20):
        r = time_forward(gen, x, single, K)
        print(json.dumps({k: v for k, v in r.items() if not k.endswith("_all")}), flush=True)
        res["forward"].append(r)
    for K in (6, 20, 64):
        r = time_summarize(K)
        print(json.dumps(r), flush=True)
        res["summarize"].append(r)
    res["wall_s"] = time.time() - t0
    with open(os.path.join(out_dir, "ensemble.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
