"""Developer tool (GPU): what gradient accumulation (TrainStep's ``accumulate_grad_batches = k``) costs on one GPU.

The bench's DN and SR-2x training workloads (F = 32, nb = 4, batch 16 of 416^2 synthetic count images, the bench's
seeded weights and loss terms) with k = 1, 2 and 4: each arm is built afresh, warmed up for two optimizer steps, then
timed over ``--steps`` optimizer steps (k micro-batches each) with CUDA events; the arms alternate, ``--rounds`` times.
Every arm cycles the same four seeded micro-batches (the first is the bench's), so the arms differ in k alone.
Prints img/s (every micro-batch's images), ms per micro-batch and torch.cuda.max_memory_allocated of the arm, after the
card's name and power limit read in the same call.

    python tools/accum_probe.py [--steps 20] [--rounds 2] [--out LOG]
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


def run(kind, k, steps, dev):
    import bench
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR
    from xmm_superres_denoise_b200.training import TrainStep
    from xmm_superres_denoise_b200.transforms import Normalize
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    b = 16
    m = (GeneratorRRDB_DN(1, 1, bench.NF, bench.NB) if kind == "dn"
         else GeneratorRRDB_SR(1, 1, bench.NF, bench.NB, num_upsample=1))
    m.load_state_dict(bench.oracle_state_dict(kind))
    m = m.to(dev).train()
    weights = {"l1": 0.5, "poisson": 0.5} if kind == "dn" else {"l1": 0.3, "poisson": 0.3, "ms_ssim": 0.4}
    step = TrainStep(m, create_loss(O.sc_dict_for("sqrt"), weights), lr=1e-4, betas=(0.9, 0.999),
                     accumulate_grad_batches=k)
    norm = Normalize(bench.LR_MAX, bench.LR_MAX if kind == "dn" else bench.HR_MAX_SR, "sqrt")
    batches = []
    for j in range(4):
        lr_np, hr_np, t_lr, t_hr = bench.synthetic_counts(b, 4321 + j, kind)
        batches.append((norm.normalize_counts(torch.from_numpy(lr_np).to(dev), norm.lr_max, exposure=t_lr),
                        norm.normalize_counts(torch.from_numpy(hr_np).to(dev), norm.hr_max, exposure=t_hr)))
    for i in range(2 * k):  # two optimizer steps
        step(*batches[i % 4])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps * k):
        loss = step(*batches[i % 4])
    e1.record()
    torch.cuda.synchronize()
    assert step.pending == 0 and step.opt.step_count == steps + 2
    ms = e0.elapsed_time(e1)
    peak = torch.cuda.max_memory_allocated(dev) - base
    val = float(loss)
    del m, step, batches
    return ms / (steps * k), b * steps * k / (ms * 1e-3), peak, val


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="optimizer steps timed per arm")
    ap.add_argument("--rounds", type=int, default=2, help="times each arm is run, arms alternating")
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
    ks = (1, 2, 4)
    for kind in ("dn", "sr"):
        res = {k: [] for k in ks}
        for r in range(args.rounds):
            for k in (ks if r % 2 == 0 else ks[::-1]):
                ms, ips, peak, val = run(kind, k, args.steps, dev)
                res[k].append((ms, ips, peak))
                say(f"{kind.upper():2s} F=32 nb=4 batch 16 k={k} round {r}: {ips:7.1f} img/s, {ms:7.3f} ms per "
                    f"micro-batch, max_memory_allocated {peak / 1e9:6.3f} GB, last loss {val:.6f}")
        for k in ks:
            ips = [v[1] for v in res[k]]
            say(f"{kind.upper():2s} k={k}: img/s mean {statistics.mean(ips):7.1f} (min {min(ips):7.1f}, max "
                f"{max(ips):7.1f}), ms per micro-batch {statistics.mean(v[0] for v in res[k]):7.3f}, peak "
                f"{max(v[2] for v in res[k]) / 1e9:6.3f} GB")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
