"""Cost of partially labelled batches (target_mask) on the B200: the DEER loss kernel pair (deer_nig_loss_stats[_mask]
+ deer_nig_loss_finish[_mask]) at B = 256 (the training size) and B = 2^22 (DESIGN.md 4.5), with and without a mask,
and the B = 256 sequence-model training step (CUDA-graph replay) without a mask, with an all-ones mask and with about
30 % of the entries unlabelled.  Variants are timed in alternating rounds with CUDA events; the card's name and power
limit are recorded with the numbers.

    python tools/target_mask_bench.py [--out profiles/target_mask_bench_b200.json] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import deer_b200  # noqa: E402
from deer_b200 import _lib, ops  # noqa: E402
from deer_b200.trainer import DEERDataParallelTrainer  # noqa: E402

DEV = "cuda"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name()}


def time_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(variants, n, rounds):
    """{name: [ms per call, one per round]} with the variants interleaved round by round."""
    for fn in variants.values():     # warm-up: module loads, occupancy queries, arena growth
        time_ms(fn, 3)
    out = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            out[k].append(time_ms(fn, n))
    return out


def summary(samples, unit_scale=1.0):
    return {k: {"median": statistics.median(v) * unit_scale, "min": min(v) * unit_scale,
                "max": max(v) * unit_scale, "rounds": [x * unit_scale for x in v]} for k, v in samples.items()}


def loss_pair(B, rounds):
    g = torch.Generator().manual_seed(B)
    nset = 2 if B * 3 * 20 > (256 << 20) else max(2, (512 << 20) // (B * 3 * 20))   # rotating sets past the 126 MB L2
    nset = min(nset, 8)
    ev = [torch.randn(B, 3, 4, generator=g).to(DEV) for _ in range(nset)]
    tg = [torch.tanh(torch.randn(B, 3, generator=g)).to(DEV) for _ in range(nset)]
    mk = [(torch.rand(B, 3, generator=g) >= 0.3).to(DEV) for _ in range(nset)]
    variants = {
        "no_mask": lambda i: ops.nig_loss_raw(ev[i % nset], None, tg[i % nset], want_nig=True, want_grad=True),
        "mask_30pct_unlabelled": lambda i: ops.nig_loss_raw(ev[i % nset], None, tg[i % nset], want_nig=True,
                                                            want_grad=True, target_mask=mk[i % nset]),
    }
    n = 200 if B <= 4096 else 20
    return {"B": B, "D": 3, "rotating_input_sets": nset, "calls_per_round": n,
            "us_per_pair": summary(alternate(variants, n, rounds), 1e3)}


def train_step(rounds):
    sys.path.insert(0, ROOT)
    from bench import synth_batch
    B = 256
    torch.manual_seed(42)
    model = deer_b200.SequenceDEERModel(dropout=0.3).to(DEV).train()
    trainer = DEERDataParallelTrainer(model, learning_rate=1e-4, weight_decay=1e-5, gradient_clip=1.0)
    gen = torch.Generator().manual_seed(1234)
    batches = {"no_mask": synth_batch(B, DEV, gen), "all_ones_mask": synth_batch(B, DEV, gen),
               "mask_30pct_unlabelled": synth_batch(B, DEV, gen)}
    batches["all_ones_mask"]["target_mask"] = torch.ones(B, 3, dtype=torch.bool, device=DEV)
    m = torch.rand(B, 3, generator=gen) >= 0.3
    batches["mask_30pct_unlabelled"]["target_mask"] = m.to(DEV)
    batches["mask_30pct_unlabelled"]["targets"][~m.to(DEV)] = float("nan")
    launches = {}
    for _ in range(2):               # the second pass: lazily created state (scratch arena, descriptors) exists
        for k, b in batches.items():
            l0 = _lib.launch_count()
            trainer.train_step(b)
            launches[k] = _lib.launch_count() - l0
    replays = {k: trainer.capture(b) for k, b in batches.items()}
    variants = {k: (lambda i, r=r: r()) for k, r in replays.items()}
    res = summary(alternate(variants, 50, rounds))
    torch.cuda.synchronize()
    finite = bool(torch.isfinite(trainer.flat.params).all())
    return {"B": B, "steps_per_round": 50, "ms_per_step": res, "launches_per_step": launches,
            "parameters_finite": finite}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "target_mask_bench_b200.json"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("target_mask_bench: needs a CUDA device")
    res = {"card": card(), "loss_pair": [loss_pair(256, args.rounds), loss_pair(1 << 22, args.rounds)],
           "train_step": train_step(args.rounds)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
