"""Developer tool (GPU): what memory-efficient training (the generator's ``memory_efficient``) costs and saves.

For DN and SR-2x at F = 32, nb = 4, batch 16, 416^2 LR: TrainStep step time (CUDA events, 20 steps after 3 warm-up
steps) and torch.cuda.max_memory_allocated of those steps, with the flag off and on.  Then one step with the flag on at
DN F = 32, nb = 23, batch 64 (BASELINE config-5 depth); with the flag off that size is not allocated, its training
buffers are computed from their shapes.  Prints the card's name and power limit first.

    python tools/memeff_probe.py [--out LOG]
"""
import argparse
import gc
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def buffer_bytes(kind, nf, nb, b, h, w, memeff, up=1):
    """Bytes of TrainEngine._train_buffers (bf16 feature maps + the fp32 pre-clamp image)."""
    plane = b * h * w * nf * 2  # one F-channel bf16 map
    n = 3 * 5 + 3  # gradient ring (5F each) + trunk, d_trunk, d_fea
    n += (3 * nb + 1) + 5 if memeff else 3 * nb * 5 + 1  # checkpoints + scratch, or every block's [x0..x4] + last output
    total = n * plane
    s = 1
    if kind == "sr":
        for _ in range(up):
            s *= 2
            total += b * (h * s) * (w * s) * nf * 2 + b * (h * s // 2) * (w * s // 2) * 4 * nf * 2  # up, d_up
        total += 2 * b * (h * s) * (w * s) * nf * 2  # hr, d_hr
    return total + b * (h * s) * (w * s) * 4


def run(kind, nf, nb, b, memeff, steps, warmup, dev):
    from oracle import rrdb_oracle as O
    from xmm_superres_denoise_b200.models import GeneratorRRDB_DN, GeneratorRRDB_SR
    from xmm_superres_denoise_b200.training import TrainStep
    from xmm_superres_denoise_b200.utils.loss_functions import create_loss

    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    h = w = 416
    s = 1 if kind == "dn" else 2
    m = GeneratorRRDB_DN(1, 1, nf, nb) if kind == "dn" else GeneratorRRDB_SR(1, 1, nf, nb, num_upsample=1)
    m.load_state_dict(O.init_state_dict(kind, 1, 1, nf, nb, 1, seed=3))
    m.memory_efficient = memeff
    m = m.to(dev).train()
    weights = {"l1": 0.5, "poisson": 0.5} if kind == "dn" else {"l1": 0.3, "poisson": 0.3, "ms_ssim": 0.4}
    step = TrainStep(m, create_loss(O.sc_dict_for("sqrt"), weights), lr=1e-4)
    g = torch.Generator().manual_seed(7)
    x = torch.rand(b, 1, h, w, generator=g).to(dev)
    t = (torch.rand(b, 1, h * s, w * s, generator=g) * 0.5).to(dev)
    for _ in range(warmup):
        step(x, t)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step(x, t)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / max(steps, 1)
    peak = torch.cuda.max_memory_allocated(dev)
    val = float(loss)
    del m, step, x, t
    return ms, peak, val


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    say(f"card: {card}")
    dev = torch.device("cuda:0")
    torch.cuda.init()
    torch.zeros(1, device=dev)  # a context before the first reset_peak_memory_stats
    gb = 1e9
    for kind in ("dn", "sr"):
        res = {}
        for memeff in (False, True):
            res[memeff] = run(kind, 32, 4, 16, memeff, args.steps, args.warmup, dev)
            ms, peak, val = res[memeff]
            say(f"{kind.upper():2s} F=32 nb=4 batch 16 memory_efficient={int(memeff)}: {ms:8.2f} ms/step "
                f"({16e3 / ms:6.1f} img/s), max_memory_allocated {peak / gb:6.2f} GB, training buffers from shapes "
                f"{buffer_bytes(kind, 32, 4, 16, 416, 416, memeff) / gb:6.2f} GB, loss {val:.6f}")
        say(f"{kind.upper():2s} F=32 nb=4 batch 16: step time x{res[True][0] / res[False][0]:.3f}, "
            f"peak memory x{res[True][1] / res[False][1]:.3f}")
    ms, peak, val = run("dn", 32, 23, 64, True, 1, 1, dev)
    say(f"DN F=32 nb=23 batch 64 memory_efficient=1: {ms:8.2f} ms/step (one step after one warm-up), "
        f"max_memory_allocated {peak / gb:6.2f} GB, training buffers from shapes "
        f"{buffer_bytes('dn', 32, 23, 64, 416, 416, True) / gb:6.2f} GB, loss {val:.6f}")
    say(f"DN F=32 nb=23 batch 64 memory_efficient=0: not allocated; training buffers from shapes "
        f"{buffer_bytes('dn', 32, 23, 64, 416, 416, False) / gb:6.2f} GB")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
