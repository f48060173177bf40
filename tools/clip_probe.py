"""Developer tool (GPU): what gradient clipping (TrainStep's ``gradient_clip_val`` / ``gradient_clip_algorithm``) costs.

1. The norm kernels (``xmm_grad_clip_coef``: per-CTA fp64 partials, then the finalize launch): ``--launches`` calls
   captured as one CUDA graph, its replay timed with CUDA events, at the DN and SR default parameter counts (F = 32, nb = 4: 1.67 M, 1.72 M) and at
   F = 64, nb = 23 (38 M): once on one buffer, which the default sizes' 6.7 MB leave resident in the 126 MB L2, and
   once cycling through copies that add up to more than twice the L2, so that every call reads HBM.  GB/s counts the
   4 bytes per gradient each call reads.  Next to it the plain Adam kernel and the clipping one at the same sizes.
2. Training img/s for the bench's DN and SR-2x workloads (F = 32, nb = 4, batch 16 of 416^2 synthetic count images,
   the bench's seeded weights and loss terms) with clipping off, by norm and by value: each arm is built afresh, warmed
   up for two steps, then timed over ``--steps`` optimizer steps with CUDA events; the arms alternate, ``--rounds``
   times.  Arms: off; by norm with max_norm above the norm (the clip's launches on the plain trajectory); by norm at
   0.5 and by value at 1e-3 (both act on every step); by value at 1e-6 (every element clamped).
The card's name and power limit are read in the same call.

    python tools/clip_probe.py [--steps 20] [--rounds 2] [--launches 200] [--out LOG]
"""
import argparse
import gc
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 2**20
# training arms: (gradient_clip_val, algorithm).  "norm-idle" clips by norm above the norm (coefficient 1: the plain
# step's trajectory with the clip's launches); "norm" / "value" clip every step, "value-all" clamps every element.
ARMS = {"off": (None, "norm"), "norm-idle": (1e30, "norm"), "norm": (0.5, "norm"), "value": (1e-3, "value"),
        "value-all": (1e-6, "value")}


def _time(fn, launches):
    """us per call of fn(i), i < launches, captured as one CUDA graph and replayed: the kernels' time without the
    ~10 us of Python and ctypes each call costs on the host."""
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(launches):
            fn(i)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / launches


def kernels(n, launches, dev, say):
    from xmm_superres_denoise_b200 import _lib, training

    copies = max(1, -(-2 * L2_BYTES // (4 * n)) + 1)
    gs = [torch.randn(n, device=dev) * 1e-3 for _ in range(copies)]
    out = torch.empty(2, device=dev)
    ws = training.grad_norm_workspace(n, dev)
    warm = _time(lambda i: training.grad_clip_coef(gs[0], 1.0, 1e-3, out, ws), launches)
    cold = _time(lambda i: training.grad_clip_coef(gs[i % copies], 1.0, 1e-3, out, ws), launches)
    gb = 4 * n / 1e9
    say(f"grad_clip_coef n={n:>9d} ({4 * n / 1e6:6.1f} MB): one buffer {warm:7.2f} us ({gb / (warm * 1e-6):6.0f} GB/s), "
        f"{copies} buffers cycled {cold:7.2f} us ({gb / (cold * 1e-6):6.0f} GB/s)")
    p, m, v = torch.zeros(n, device=dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    lib = _lib.load()
    plain = _time(lambda i: lib.xmm_adam_step(p.data_ptr(), gs[0].data_ptr(), m.data_ptr(), v.data_ptr(), n, 1e-4,
                                              0.9, 0.999, 1e-8, 1 + i, 1.0, _lib.stream_ptr()), launches)
    clip_n = _time(lambda i: lib.xmm_adam_step_clip(p.data_ptr(), gs[0].data_ptr(), m.data_ptr(), v.data_ptr(), n,
                                                    1e-4, 0.9, 0.999, 1e-8, 1 + i, 1.0, out.data_ptr() + 4, 0.0,
                                                    _lib.stream_ptr()), launches)
    clip_v = _time(lambda i: lib.xmm_adam_step_clip(p.data_ptr(), gs[0].data_ptr(), m.data_ptr(), v.data_ptr(), n,
                                                    1e-4, 0.9, 0.999, 1e-8, 1 + i, 1.0, None, 1e-3,
                                                    _lib.stream_ptr()), launches)
    say(f"adam n={n:>9d}: plain {plain:7.2f} us, clip by norm {clip_n:7.2f} us, clip by value {clip_v:7.2f} us "
        f"(one buffer, {28 * n / 1e9 / (plain * 1e-6):6.0f} GB/s at 28 B per parameter for the plain step)")
    del gs, p, m, v


def train(kind, clip, steps, dev):
    import bench
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR
    from xmm_superres_denoise_b200.training import TrainStep
    from xmm_superres_denoise_b200.transforms import Normalize
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    gc.collect()
    torch.cuda.empty_cache()
    b = 16
    m = (GeneratorRRDB_DN(1, 1, bench.NF, bench.NB) if kind == "dn"
         else GeneratorRRDB_SR(1, 1, bench.NF, bench.NB, num_upsample=1))
    m.load_state_dict(bench.oracle_state_dict(kind))
    m = m.to(dev).train()
    weights = {"l1": 0.5, "poisson": 0.5} if kind == "dn" else {"l1": 0.3, "poisson": 0.3, "ms_ssim": 0.4}
    val, algorithm = ARMS[clip]
    step = TrainStep(m, create_loss(O.sc_dict_for("sqrt"), weights), lr=1e-4, betas=(0.9, 0.999),
                     gradient_clip_val=val, gradient_clip_algorithm=algorithm)
    norm = Normalize(bench.LR_MAX, bench.LR_MAX if kind == "dn" else bench.HR_MAX_SR, "sqrt")
    lr_np, hr_np, t_lr, t_hr = bench.synthetic_counts(b, 4321, kind)
    x = norm.normalize_counts(torch.from_numpy(lr_np).to(dev), norm.lr_max, exposure=t_lr)
    y = norm.normalize_counts(torch.from_numpy(hr_np).to(dev), norm.hr_max, exposure=t_hr)
    for _ in range(2):
        step(x, y)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step(x, y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    gn = None if step.grad_norm is None else float(step.grad_norm)
    val = float(loss)
    del m, step
    return ms / steps, b * steps / (ms * 1e-3), val, gn


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="optimizer steps timed per arm")
    ap.add_argument("--rounds", type=int, default=2, help="times each arm is run, arms alternating")
    ap.add_argument("--launches", type=int, default=200, help="calls timed per kernel measurement")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    say(f"card: {card}")
    dev = torch.device("cuda:0")
    torch.zeros(1, device=dev)
    for n in (1670657, 1716897, 38214465):  # DN / SR F=32 nb=4, DN F=64 nb=23
        kernels(n, args.launches, dev, say)
    arms = tuple(ARMS)
    for kind in ("dn", "sr"):
        res = {a: [] for a in arms}
        for r in range(args.rounds):
            for a in (arms if r % 2 == 0 else arms[::-1]):
                ms, ips, val, gn = train(kind, a, args.steps, dev)
                res[a].append((ms, ips))
                say(f"{kind.upper():2s} F=32 nb=4 batch 16 clip={a:9s} round {r}: {ips:7.1f} img/s, {ms:7.3f} ms per "
                    f"step, last loss {val:.6f}" + ("" if gn is None else f", grad_norm {gn:.5g}"))
        for a in arms:
            ips = [v[1] for v in res[a]]
            say(f"{kind.upper():2s} clip={a:9s}: img/s mean {statistics.mean(ips):7.1f} (min {min(ips):7.1f}, max "
                f"{max(ips):7.1f}), ms per step {statistics.mean(v[0] for v in res[a]):7.3f}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
