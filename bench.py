#!/usr/bin/env python
"""bench.py - DEER hot-path benchmark (BASELINE.json metric: train-step and inference samples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the hot path over one synthetic batch of the BASELINE shapes
(audio [B,300,84], video [B,50,256], text [B,64,768], mask, linguistic features, targets [B,3]):
  * headline `value`: TRAINING step (forward + DEER multitask loss + backward + gradient all-reduce + clip + AdamW),
    B=256 per GPU (BASELINE configs[2]; configs[3] at N>1, weak scaling), inputs resident in HBM;
  * `inference`: eval/no-grad forward, B=1024 per GPU (BASELINE configs[1]);
  * `e2e`: the same training step driven through the public trainer API from PINNED HOST buffers, H2D copies and the
    D2H loss read inside the timed region;
  * `roofline`: the dominant kernel timed alone with CUDA events;
  * `cpu_baseline`: the stock-torch.nn CPU port of the reference path (oracle/torch_baseline.py) on a bounded sample.
Prints ONE JSON line on rank 0.  The training, e2e, strong-scaling and inference loops each time exactly K steps.

--dump-outputs DIR (rank 0) writes what the last timed training step computed, as float32 DIR/<name>.npy.  Inputs,
weights and dropout masks are seeded, so two builds run with the same arguments can be compared file for file, within
the run-to-run spread given in dump_outputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the checkout it runs from untouched (it may be read-only)

TRAIN_B, INFER_B = 256, 1024
TA, TV, TT = 300, 50, 64
# algorithmic work per sample (SURVEY.md section 8d)
FWD_FLOP_PER_SAMPLE = 1.673e9
TRAIN_FLOP_PER_SAMPLE = 3 * FWD_FLOP_PER_SAMPLE
INPUT_BYTES_PER_SAMPLE = (TA * 84 + TV * 256 + TT * 768 + TT + 10 + 3) * 4


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[4:8]):
                    if "Active" in v and "Not" not in v:
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def synth_batch(B, device, gen, pinned=False):
    import torch
    kw = dict(generator=gen)
    audio = torch.randn(B, TA, 84, **kw)
    video = torch.randn(B, TV, 256, **kw)
    text = torch.randn(B, TT, 768, **kw)
    mask = torch.ones(B, TT)
    ling = torch.zeros(B, 10)
    y = torch.tanh(torch.randn(B, 3, **kw) + 0.1 * torch.randn(B, 3, **kw))
    b = {"audio_features": audio, "video_features": video, "text_features": text, "attention_mask": mask,
         "linguistic_features": ling, "targets": y}
    if pinned:
        return {k: v.pin_memory() for k, v in b.items()}
    return {k: v.to(device) for k, v in b.items()}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path.  /root/reference is pure Python and does not
    travel to the GPU box, so the stock-torch.nn port in oracle/torch_baseline.py (checked against the golden-pinned
    oracle) is what runs, with every host thread, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import torch_baseline as TB
    sample_b = args.ref_batch       # default: the SAME batch as the GPU arm (B=256, ~3 s per step on 16 host threads)
    sps, dt, threads = TB.time_cpu_baseline("train", sample_b, iters=max(1, args.steps), warmup=max(1, args.warmup))
    line = {
        "impl": "reference", "metric": "deer_train_step_samples_per_s", "value": sps, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "same_config": sample_b == TRAIN_B,
        "config": {"workload": f"sequence DEER train step (fwd+loss+bwd+clip+AdamW) on host CPU, B={sample_b} per step "
                               f"(GPU arm: B={TRAIN_B}/GPU); audio {TA}x84, video {TV}x256, text {TT}x768, dropout 0.3",
                   "batch_per_step": sample_b},
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port",
                         "sample": f"B={sample_b} train steps x{args.steps} (oracle/torch_baseline.py: stock torch.nn "
                                   "layers wired as the reference wires them; /root/reference cannot travel)"},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-pooled", action="store_true")
    ap.add_argument("--no-text-stream", action="store_true", help="ablation: text encoder on the video encoder's stream")
    ap.add_argument("--no-pool-rowterm", action="store_true", help="ablation: pooling input gradient written by the pooling kernel, the scorer GEMM accumulates onto it")
    ap.add_argument("--lstm-defer-wgrad", action="store_true", help="ablation: LSTM layer-1 weight gradients on the weight-gradient stream instead of in front of layer 0's BPTT (measured: no gain)")
    ap.add_argument("--no-branch-streams", action="store_true",
                    help="ablation: video/text encoders on the main stream behind the audio encoder")
    ap.add_argument("--overlap-exchange", action="store_true",
                    help="ablation: all-reduce the non-audio gradients beside the audio backward (measured: no gain)")
    ap.add_argument("--exchange-ctas", type=int, default=None,
                    help="CTA limit of the NCCL communicator of the overlapped gradient buckets (default 8)")
    ap.add_argument("--branch-max-batch", type=int, default=None)
    ap.add_argument("--tf32-pair", type=int, default=None, help="DEER_OPT_TF32_PAIR override (ablation)")
    ap.add_argument("--lstm-dual", type=int, default=None, help="DEER_OPT_LSTM_DUAL override (ablation)")
    ap.add_argument("--lstm-tile", type=int, default=None, help="DEER_OPT_LSTM_TILE override (ablation)")
    ap.add_argument("--lstm-halfsplit", type=int, default=None, help="DEER_OPT_LSTM_HALFSPLIT override (ablation)")
    ap.add_argument("--lstm-stasync", type=int, default=None, help="DEER_OPT_LSTM_STASYNC override (ablation)")
    ap.add_argument("--lstm-xin", type=int, default=None, help="DEER_OPT_LSTM_XIN override (ablation): 0 = layer-0 input projection as a GEMM")
    ap.add_argument("--chain", action="store_true",
                    help="ablation: fusion + head as the persistent chain kernel (one launch per direction; measured slower)")
    ap.add_argument("--train-only", action="store_true", help="ablation runs: only the training-step line (no e2e / inference / roofline)")
    ap.add_argument("--no-defer-wgrad", action="store_true",
                    help="ablation: small-layer weight gradients on the main stream")
    ap.add_argument("--ref-batch", type=int, default=TRAIN_B, help="batch of the CPU reference arm (default: same as GPU)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="STRONG scaling: fixed global batch split over the ranks (BASELINE configs[3]: 2048); the "
                         "headline then reports scaling=strong.  Default 0: weak scaling, B=256 per GPU")
    ap.add_argument("--no-strong", action="store_true", help="skip the extra strong-scaling block (global batch 2048)")
    ap.add_argument("--no-loss-check", action="store_true", help="skip the step-0 loss check against the CPU port")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path; the reference arm has no such dump")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import deer_b200
    from deer_b200 import _lib, ops
    from deer_b200.trainer import DEERDataParallelTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, args.warmup
    pk = peaks()
    ops.set_branch_streams(not args.no_branch_streams)
    ops.set_text_stream(not args.no_text_stream)
    ops.set_pool_rowterm(not args.no_pool_rowterm)
    ops.set_lstm_defer_wgrad(args.lstm_defer_wgrad)
    ops.set_defer_wgrad(not args.no_defer_wgrad)
    if args.branch_max_batch is not None:
        ops.set_branch_max_batch(args.branch_max_batch)
    if args.lstm_dual is not None:
        _lib.set_option(9, args.lstm_dual)
    if args.lstm_tile is not None:
        _lib.set_option(3, args.lstm_tile)
    if args.lstm_halfsplit is not None:
        _lib.set_option(13, args.lstm_halfsplit)
    if args.lstm_stasync is not None:
        _lib.set_option(12, args.lstm_stasync)
    if args.lstm_xin is not None:
        _lib.set_option(15, args.lstm_xin)
    if args.chain:
        from deer_b200 import chain as _chain
        _chain.set_enabled(True)
    if args.tf32_pair is not None:
        _lib.set_option(6, args.tf32_pair)
        if not args.tf32_pair:
            ops.set_conv_window(False)   # the sliding-window Conv1d needs the pair kernel's TMA reduce epilogue

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ------------------------------------------------------------------ model + trainer
    strong = args.global_batch > 0
    if strong and args.global_batch % world:
        raise SystemExit(f"--global-batch {args.global_batch} is not divisible by {world} ranks")
    B = args.global_batch // world if strong else TRAIN_B
    torch.manual_seed(42)
    model = deer_b200.SequenceDEERModel(dropout=0.3).to(dev).train()
    trainer = DEERDataParallelTrainer(model, learning_rate=1e-4, weight_decay=1e-5, gradient_clip=1.0)
    if args.exchange_ctas is not None:
        trainer.exchange_ctas = args.exchange_ctas
    gen = torch.Generator().manual_seed(1234 + rank)
    use_graph = not args.no_graph

    # step-0 check of the path being timed against the CPU port (same weights, same inputs; eval mode so that neither
    # side draws dropout masks): the loss the bench optimises is the reference's loss
    loss_check = None
    if rank == 0 and not args.no_loss_check:
        loss_check = check_loss_against_port(torch, model, dev, gen)

    def measure_train(Bt, steps, warm):
        """(ms per step, launches per step, final loss) of the trainer step at Bt samples per GPU, inputs resident."""
        nb = max(2, min(4, (256 * 4) // Bt))    # rotating resident batches: >= 2, 4 x 89 MB at B=256 (> 126 MB L2)
        batches = [synth_batch(Bt, dev, gen) for _ in range(nb)]
        trainer.train_step(batches[0])
        l0 = _lib.launch_count()
        trainer.train_step(batches[0])
        launches = _lib.launch_count() - l0
        # the whole step (fwd + loss + bwd + all-reduce + clip + AdamW) captured once per resident batch and replayed
        replays = [trainer.capture(b) for b in batches] if use_graph else None

        def fn(i):
            if use_graph:
                replays[i % nb]()
            else:
                trainer.train_step(batches[i % nb])

        for i in range(warm):
            fn(i)
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ms = timed(fn, steps)
        clk = sampler.stop() if rank == 0 else None
        return ms / steps, launches, float(trainer.last_losses[-1]), clk, nb

    overlap_check = None
    if world > 1:
        # the early (overlapped) gradient exchange must give the same reduced gradients as one all-reduce at the end,
        # up to the run-to-run noise of the atomically accumulated / split-K gradients (measured on the spot)
        b0 = synth_batch(B, dev, gen)
        g = []
        for ov in (True, False, False):
            trainer.overlap_exchange = ov
            trainer.forward_backward(b0)
            if not trainer._grads_reduced:
                trainer._allreduce(trainer.flat.grads)
            trainer._grads_reduced = False
            torch.cuda.synchronize()
            g.append(trainer.flat.grads.clone())
        trainer.overlap_exchange = args.overlap_exchange
        noise = float((g[1] - g[2]).norm() / g[2].norm())
        overlap_check = float((g[0] - g[2]).norm() / g[2].norm())
        assert overlap_check < 3 * noise + 1e-5, f"overlapped gradient exchange differs: {overlap_check} (noise {noise})"
        del g, b0

    ms_per_step, launches_per_step, final_loss, clocks, NB = measure_train(B, K, W)
    value = B * world / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, {"train_losses": trainer.last_losses, "train_params": trainer.flat.params})
    if args.train_only:
        if rank == 0:
            print(json.dumps({"metric": "deer_train_step_samples_per_s", "value": value, "ms_per_step": ms_per_step,
                              "launches_per_step": int(launches_per_step), "ablation": vars(args)}), flush=True)
        if world > 1:
            teardown_distributed(torch, dist, trainer)
        return

    # ------------------------------------------------------------------ e2e: pinned host -> device every step
    # Public API path: pinned host batch -> deer_b200.data.DevicePrefetcher (H2D on a copy stream into rotating static
    # device buffers) -> trainer step (graph replay on that buffer set) -> D2H read of the loss, every step inside the
    # timed region.  The copy of step i+1 runs while step i computes; every byte still crosses PCIe per step.
    from deer_b200.data import DevicePrefetcher
    host = [synth_batch(B, None, gen, pinned=True) for _ in range(2)]
    stager = DevicePrefetcher([], dev, depth=2)
    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]     # pinned landing buffers for the per-step loss
    loss_done = [torch.cuda.Event() for _ in range(2)]
    loss_log = []
    state = {"next": stager.stage(host[0]), "i": 0}

    def e2e_fn(_):
        i = state["i"]
        state["i"] = i + 1
        j = i % 2
        cur = state["next"]
        state["next"] = stager.stage(host[(i + 1) % 2])      # prefetch the next step's batch
        stager.wait(cur)
        tens = stager.tensors(cur)
        losses = (trainer.train_step_auto(tens, eager_steps=1, static_inputs=True) if use_graph
                  else trainer.train_step(tens))
        stager.release(cur)
        # D2H read of the step's loss: asynchronous copy into pinned memory every step; the host consumes the value
        # one step later (after its event), so kernel launches of step i+1 are never held back by a device sync
        loss_host[j].copy_(losses[-1:], non_blocking=True)
        loss_done[j].record()
        if i > 0:
            loss_done[1 - j].synchronize()
            loss_log.append(float(loss_host[1 - j]))

    for i in range(6):        # per buffer set: one eager step, then the capture; afterwards replays only
        e2e_fn(i)
    torch.cuda.synchronize()
    h2d = stager.bytes_per_batch
    e2e_ms = timed(e2e_fn, K) / K
    e2e_value = B * world / (e2e_ms / 1e3)
    torch.cuda.synchronize()
    assert len(loss_log) >= K and all(v == v for v in loss_log[-K:]), "e2e loop must deliver a finite loss every step"
    del host

    # ------------------------------------------------------------------ strong scaling (BASELINE configs[3]): global 2048
    strong_block = None
    if not strong and not args.no_strong and STRONG_GLOBAL % world == 0:
        Bs = STRONG_GLOBAL // world
        if Bs == B:
            strong_block = {"global_batch": STRONG_GLOBAL, "batch_per_gpu": Bs, "value": value,
                            "ms_per_step": ms_per_step, "unit": "samples/s", "note": "same run as the headline"}
        else:
            sms, _, _, _, _ = measure_train(Bs, K, 3)
            strong_block = {"global_batch": STRONG_GLOBAL, "batch_per_gpu": Bs, "value": STRONG_GLOBAL / (sms / 1e3),
                            "ms_per_step": sms, "unit": "samples/s", "steps": K}
        trainer._graphs.clear()
        torch.cuda.empty_cache()

    # ------------------------------------------------------------------ inference B=1024
    model.eval()
    ibatches = [synth_batch(INFER_B, dev, gen) for _ in range(2)]
    ikeys = ("audio_features", "video_features", "text_features", "attention_mask", "linguistic_features")

    def infer_eager(b):
        with torch.no_grad():
            return model(*[b[k] for k in ikeys])

    for i in range(2):
        infer_eager(ibatches[i])
    l0 = _lib.launch_count()
    infer_eager(ibatches[0])
    infer_launches = _lib.launch_count() - l0
    from deer_b200.trainer import capture_forward
    if use_graph:
        ireplays = [capture_forward(model, *[b[k] for k in ikeys])[0] for b in ibatches]

    def infer_fn(i):
        if use_graph:
            ireplays[i % 2]()
        else:
            infer_eager(ibatches[i % 2])

    infer_ms = timed(infer_fn, K) / K
    infer_value = INFER_B * world / (infer_ms / 1e3)
    del ibatches
    # inference end to end: pinned host batch (357 MB at B=1024) -> H2D -> forward -> D2H of the NIG parameters
    ihost = [{k: v for k, v in synth_batch(INFER_B, None, gen, pinned=True).items() if k in ikeys} for _ in range(2)]
    istager = DevicePrefetcher([], dev, depth=2)
    nig_host = [torch.zeros(4, INFER_B, 3).pin_memory() for _ in range(2)]
    istate = {"next": istager.stage(ihost[0]), "i": 0, "replays": {}}

    def infer_e2e(_):
        i = istate["i"]
        istate["i"] = i + 1
        cur = istate["next"]
        istate["next"] = istager.stage(ihost[(i + 1) % 2])
        istager.wait(cur)
        tens = istager.tensors(cur)
        key = tens["audio_features"].data_ptr()
        if use_graph and key not in istate["replays"]:
            istate["replays"][key] = capture_forward(model, *[tens[k] for k in ikeys])
        if use_graph:
            rep, out = istate["replays"][key]
            rep()
        else:
            out = infer_eager(tens)
        istager.release(cur)
        dst = nig_host[i % 2]
        for q, k in enumerate(("gamma", "nu", "alpha", "beta")):
            dst[q].copy_(out[k], non_blocking=True)

    for i in range(3):
        infer_e2e(i)
    torch.cuda.synchronize()
    infer_e2e_ms = timed(infer_e2e, K) / K
    torch.cuda.synchronize()
    assert bool(torch.isfinite(nig_host[0]).all())
    infer_h2d = istager.bytes_per_batch
    model.train()
    del ihost, istate, istager
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ roofline of the dominant kernels
    roof = roofline_probe(torch, ops, dev, pk)

    # ------------------------------------------------------------------ BASELINE configs[4]: pooled CompleteDEERModel on
    # multi-dataset-shaped batches (84/256/768-D vectors + targets[3] + dataset_id), batch sweep, train step + inference
    pooled = (pooled_sweep(torch, deer_b200, DEERDataParallelTrainer, dev, use_graph)
              if (world == 1 and not args.no_pooled) else None)

    inference = {"value": infer_value, "unit": "samples/s", "batch_per_gpu": INFER_B, "ms_per_step": infer_ms,
                 "launches_per_step": int(infer_launches),
                 "tensor_frac_of_sustained_bf16": infer_value / world * FWD_FLOP_PER_SAMPLE / 1e12 /
                 pk["bf16_tflops_sustained"],
                 "e2e": {"value": INFER_B * world / (infer_e2e_ms / 1e3), "unit": "samples/s",
                         "ms_per_step": infer_e2e_ms, "h2d_bytes_per_step": infer_h2d,
                         "d2h_bytes_per_step": 4 * INFER_B * 3 * 4,
                         "note": "PCIe-bound: 357 MB of fp32 features per forward"}}
    line = {
        "metric": "deer_train_step_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if strong else "weak",
        "vs_baseline": None,
        "dtype": "mixed: fp16/bf16 (LSTM GEMMs + recurrence) and tf32 (scorers, conv, projections) tensor-core operands, "
                 "fp32 accumulate; 3xTF32 (fp32-grade) fusion/head chain; fp32 transcendentals and loss",
        "data": "synthetic",
        "config": {"workload": f"sequence DEER training step: fwd + DEER multitask NIG loss + bwd + grad all-reduce + "
                               f"clip + AdamW; B={B}/GPU (global {B * world}), audio {TA}x84, video "
                               f"{TV}x256, text {TT}x768, dropout 0.3, 9,262,642 params",
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2_policy": f"{NB} rotating resident input batches ({NB * B * INPUT_BYTES_PER_SAMPLE / 1e6:.0f} "
                                "MB) + >1 GB of activations per step, larger than the 126 MB L2",
                   "loss_semantics": "exact global batch (loss statistics all-reduced)", "final_loss": final_loss,
                   "loss_check_vs_cpu_port": loss_check},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "api": "deer_b200.data.DevicePrefetcher -> DEERDataParallelTrainer.train_step_auto"},
        "cuda_graph": use_graph, "branch_streams": ops.branch_streams_enabled(),
        "exchange_overlap": bool(world > 1 and trainer.overlap_exchange), "exchange_overlap_check": overlap_check,
        "gpu_launches": int(launches_per_step * K),
        "launches_per_step": int(launches_per_step),
        "inference": inference,
        "strong_scaling": strong_block,
        "train_tensor_frac_of_sustained_bf16": value / world * TRAIN_FLOP_PER_SAMPLE / 1e12 / pk["bf16_tflops_sustained"],
        "roofline": roof,
        "peaks": pk,
    }
    # (the driver's parser keeps nested keys of `config` / `e2e` / `roofline`: the inference and strong-scaling numbers are
    # mirrored there so they survive into BENCH_rNN.json / SCALE_rNN.json)
    line["config"]["inference"] = {k: inference[k] for k in ("value", "ms_per_step", "batch_per_gpu")}
    line["config"]["inference"]["e2e_value"] = inference["e2e"]["value"]
    line["config"]["strong_scaling"] = strong_block
    roof["inference"] = inference
    if pooled is not None:
        line["pooled_model_sweep"] = pooled
        line["config"]["pooled_model_sweep"] = pooled
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import torch_baseline as TB
        sb = TRAIN_B
        sps, dt, threads = TB.time_cpu_baseline("train", sb, iters=3, warmup=1)
        sps32, dt32, _ = TB.time_cpu_baseline("train", 32, iters=4, warmup=1)
        isps, idt, _ = TB.time_cpu_baseline("infer", 256, iters=3, warmup=1)
        line["cpu_baseline"] = {"value": sps, "unit": "samples/s", "cores": threads, "kind": "port",
                                "sample": f"B={sb} train steps x3 ({dt:.2f} s/step): the same per-step workload as the GPU "
                                          "arm; oracle/torch_baseline.py (stock torch.nn, oneDNN LSTM)",
                                "value_b32": sps32, "sample_b32": f"B=32 x4 ({dt32:.2f} s/step)",
                                "inference_value": isps, "inference_sample": f"B=256 x3 ({idt:.2f} s/step)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        teardown_distributed(torch, dist, trainer)


STRONG_GLOBAL = 2048


def teardown_distributed(torch, dist, trainer):
    """Leave a multi-rank run: drop the captured graphs (they hold NCCL work), drain, meet the other ranks, destroy the
    process group.  destroy_process_group after graph-captured collectives hung at exit on NCCL 2.28 in round 1, so it
    runs under a watchdog: if it has not returned after 20 s the rank leaves with os._exit(0) (all results are already
    printed and flushed)."""
    import gc
    trainer._graphs.clear()
    trainer._auto.clear()
    gc.collect()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    done = threading.Event()

    def watchdog():
        if not done.wait(20.0):
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    dist.destroy_process_group()
    done.set()


def check_loss_against_port(torch, model, dev, gen, Bc=16):
    """The GPU path's DEER multitask loss on a small batch vs the stock-torch.nn CPU port with the SAME weights
    (eval mode: no dropout masks on either side).  Asserts 1e-3 relative agreement; returns the two numbers."""
    from oracle import torch_baseline as TB
    was = model.training
    model.eval()
    b = synth_batch(Bc, "cpu", gen)
    port = TB.SequenceBaseline(dropout=0.0).eval()
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    missing, unexpected = port.load_state_dict(sd, strict=False)
    assert not missing, f"CPU port is missing weights: {missing[:4]}"
    with torch.no_grad():
        pred = port(b["audio_features"], b["video_features"], b["text_features"], b["attention_mask"],
                    b["linguistic_features"])
        ref = float(TB.multitask_loss(pred, b["targets"]))
        db = {k: v.to(dev) for k, v in b.items()}
        out = model(db)
        got = float(model.compute_loss(out, db["targets"])["total_loss"])
    model.train(was)
    rel = abs(got - ref) / max(abs(ref), 1e-12)
    assert rel <= 1e-3, f"bench loss check failed: GPU {got} vs CPU port {ref} (rel {rel:.2e})"
    return {"gpu": got, "cpu_port": ref, "rel_err": rel, "batch": Bc}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(torch, path, arrays):
    """Write {name: tensor} as float32 path/<name>.npy.

    The benchmark dumps what the last timed training step hands its caller: `train_losses`, the loss vector the step
    returns, and `train_params`, every parameter after the step's AdamW update (the trainer's flat buffer, 37 MB).
    Gradients and the inference outputs are left out: reductions that accumulate with atomics make the gradients of
    two runs differ by ~1e-4 after one step, and the 10 + W + K training steps in front of the dump amplify that until
    those arrays no longer correlate between two runs of the same build.  AdamW moves a parameter by at most ~lr per
    step, so the dumped arrays stay close: two runs of one build with --steps 20 differed by 6e-3 (parameters) and
    1.3e-2 (losses) relative to their norm (NVIDIA B200, 1000 W power limit)."""
    import numpy as np
    torch.cuda.synchronize()
    host = {k: v.detach().to("cpu", torch.float32).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT_BYTES}"
    os.makedirs(path, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(path, k + ".npy"), a)


def pooled_sweep(torch, deer_b200, Trainer, dev, use_graph=True, batches=(64, 256, 1024, 4096, 16384, 65536)):
    """Pooled-feature model (complete_project.py:462, 3,918,324 parameters): samples/s of the trainer step and of the
    eval forward per batch size (inputs resident; 5 timed steps each)."""
    torch.manual_seed(7)
    model = deer_b200.CompleteDEERModel(deer_b200.ModelConfig()).to(dev).train()
    tr = Trainer(model, learning_rate=1e-4, weight_decay=1e-5, gradient_clip=1.0)
    out = []
    for Bp in batches:
        g = torch.Generator().manual_seed(Bp)
        batch = {"audio_features": torch.randn(Bp, 84, generator=g).to(dev),
                 "video_features": torch.randn(Bp, 256, generator=g).to(dev),
                 "text_features": torch.randn(Bp, 768, generator=g).to(dev),
                 "targets": torch.tanh(torch.randn(Bp, 3, generator=g)).to(dev)}
        model.train()
        step = tr.capture(batch) if use_graph else (lambda: tr.train_step(batch))
        us_t = _time_launches(torch, lambda i: step(), 10, warm=2)
        model.eval()
        if use_graph:
            from deer_b200.trainer import capture_forward
            fwd = capture_forward(model, batch)[0]
        else:
            fwd = lambda: model(batch)  # noqa: E731
        with torch.no_grad():
            us_i = _time_launches(torch, lambda i: fwd(), 10, warm=2)
        out.append({"batch": Bp, "train_samples_per_s": Bp / (us_t * 1e-6), "train_ms": us_t / 1e3,
                    "infer_samples_per_s": Bp / (us_i * 1e-6), "infer_ms": us_i / 1e3})
    return out


def _time_launches(torch, fn, n, warm=5):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n   # us per launch


# bytes of kept BPTT state per (sample, step, direction, hidden unit): 4 activated gates + the cell state
LSTM_KEEP_BYTES_PER_UNIT = 4 * 2 + 2     # FP16 kept state (DEER_OPT_LSTM_KEEP16 = 1, default)
# dram__bytes_read.sum + dram__bytes_write.sum per launch: OFFLINE constants transcribed from the committed
# `ncu --set full` captures under profiles/ (a bench run cannot measure DRAM traffic itself; a number taken under the
# profiler is never a bench value) -- reported as `traffic` with `traffic_source`
NCU_TRAFFIC_SOURCE = ("offline ncu --set full captures of this build (dram__bytes_read.sum + dram__bytes_write.sum per launch): "
                      "profiles/r2_ncu_full_roofline_summary.txt, profiles/r2_ncu_full_lstm_summary.txt")
NCU_TRAFFIC = {
    # profiles/r2_ncu_full_roofline_summary.txt (ncu --set full --clock-control none, per launch)
    "gemm_h16_pair_out16": 80.8e6 + 255.5e6,                       # algorithmic 395 MB; part of C16 still in L2 at kernel end
    "nig_stats_plus_finish": 251.7e6 + 296.8e6 + 251.7e6 + 156.7e6,  # two passes: the 252 MB of operands are read twice
    # profiles/r2_ncu_full_lstm_summary.txt: the kernels inside the real training step (B=256, layer 1)
    "lstm_fwd_keep": 316.7e6 + 572.0e6,    # reads = the 315 MB of FP16 pre-activations; algorithmic 944 MB (tail of the stores in L2)
    "lstm_bwd": 556.3e6 + 260.0e6,         # algorithmic 865 MB
}


def roofline_probe(torch, ops, dev, pk):
    """Kernels timed alone with CUDA events on the launching stream (operands rotate through buffers larger than L2).

    Headline = the dense-contraction engine of the training step (16-bit tcgen05 GEMM) on its largest instance: the
    time-batched layer-1 LSTM input projection of both directions, gates[B*T,2048] = h0[B*T,512] W_ih^T.
    Extra entries: the fused NIG head+loss kernels at a size where HBM traffic dominates (north-star target: fraction
    of HBM peak) and the persistent LSTM recurrence (latency-bound: us per step)."""
    B, T, H = TRAIN_B, TA, 256
    M, N, K = B * T, 8 * H, 2 * H     # both directions in one contraction: pre[T*B, 2*4H] = h0[T*B, 512] W_ih^T
    nbuf = 3   # 3 x (79 MB A + 315 MB C16 [+ 629 MB fp32 C]) > 126 MB L2
    A = [(torch.randn(M, K, device=dev) * 0.5).half() for _ in range(nbuf)]
    W = (torch.randn(N, K, device=dev) * 0.05).half()
    bias = torch.randn(N, device=dev)
    C16 = [torch.empty(M, N, device=dev, dtype=torch.float16) for _ in range(nbuf)]

    def gemm_launch(i):   # exactly the call ops._BiLSTMLayerCluster.forward makes for layer 1
        j = i % nbuf
        ops.gemm_h16(A[j], K, 0, W, K, 1, None, 0, M, N, K, bias=bias, C16=C16[j], ldc16=N)

    us = _time_launches(torch, gemm_launch, 12)
    flop = 2.0 * M * N * K
    achieved = flop / (us * 1e-6) / 1e12
    alg_bytes = float(M * K * 2 + N * K * 2 + M * N * 2)
    # With the FP16 output the algorithmic traffic (A + W read once, C16 written once: 395 MB) needs 60 us at the
    # measured HBM peak, the FLOPs need 99 us at the measured bf16 peak: the binding roof is the tensor pipe (with an
    # fp32 output the same contraction was HBM-bound: 710 MB, 108 us; that variant is reported next to it).
    hbm_floor_us = alg_bytes / (pk["hbm_gbs"] * 1e3)
    tensor_floor_us = flop / (pk["bf16_tflops"] * 1e6)
    gbs = alg_bytes / (us * 1e-6) / 1e9
    hbm_bound = hbm_floor_us >= tensor_floor_us
    roof = {"kernel": "h16::gemm_h16_pair_kernel<2,0,0> (layer-1 LSTM input projection of both directions, "
                      "[76800,512]x[2048,512]^T, FP16 operands, fp32 accumulate, bias epilogue, FP16 output through "
                      "64-column TMA-store tiles; cta_group::2)",
            "bound": "hbm" if hbm_bound else "tensor",
            "achieved": gbs if hbm_bound else achieved, "peak": pk["hbm_gbs"] if hbm_bound else pk["bf16_tflops"],
            "unit": "GB/s" if hbm_bound else "TFLOP/s",
            "frac": (gbs / pk["hbm_gbs"]) if hbm_bound else (achieved / pk["bf16_tflops"]),
            "traffic": NCU_TRAFFIC.get("gemm_h16_pair_out16"), "traffic_source": NCU_TRAFFIC_SOURCE, "us_per_launch": us,
            "flop_per_launch": flop, "algorithmic_bytes_per_launch": alg_bytes,
            "hbm_floor_us": hbm_floor_us, "tensor_floor_us": tensor_floor_us,
            "hbm": {"achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"]},
            "tensor": {"achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                       "frac": achieved / pk["bf16_tflops"]},
            "peak_source": f"{pk['source']} HBM copy bandwidth / cuBLAS bf16 burst (MEASURED_PEAKS.json)"}
    del C16
    C = [torch.empty(M, N, device=dev) for _ in range(nbuf)]
    us32o = _time_launches(torch, lambda i: ops.gemm_h16(A[i % nbuf], K, 0, W, K, 1, C[i % nbuf], N, M, N, K, bias=bias), 8)
    b32 = float(M * K * 2 + N * K * 2 + M * N * 4)
    roof["fp32_output_same_shape"] = {"us_per_launch": us32o, "bound": "hbm", "algorithmic_bytes_per_launch": b32,
                                      "achieved": b32 / (us32o * 1e-6) / 1e9, "unit": "GB/s",
                                      "frac": b32 / (us32o * 1e-6) / 1e9 / pk["hbm_gbs"],
                                      "tflops": flop / (us32o * 1e-6) / 1e12}
    # the other instances of the same engine in the step (small outputs: tensor-bound)
    others = {}
    G2, In = 8 * H, 2 * H
    dpre16 = (torch.randn(M, G2, device=dev) * 0.05).bfloat16()
    wb16 = (torch.randn(G2, In, device=dev) * 0.05).bfloat16()
    xb16 = (torch.randn(M, In, device=dev) * 0.5).bfloat16()
    dx = torch.empty(M, In, device=dev)
    dw = torch.zeros(G2, In, device=dev)
    t = _time_launches(torch, lambda i: ops.gemm_h16(dpre16, G2, 0, wb16, In, 0, dx, In, M, In, G2, a_bf16=True,
                                                    b_bf16=True), 8)
    others["dx [76800,2048]x[2048,512] (bf16)"] = {"us_per_launch": t, "achieved": 2.0 * M * In * G2 / t / 1e6,
                                                   "unit": "TFLOP/s", "frac": 2.0 * M * In * G2 / t / 1e6 / pk["bf16_tflops"]}
    t = _time_launches(torch, lambda i: ops.gemm_h16(dpre16, G2, 1, xb16, In, 0, dw, In, G2, In, M, a_bf16=True,
                                                    b_bf16=True, beta=1.0), 8)
    others["dW_ih [76800,2048]^T x [76800,512] (bf16, split-K)"] = {
        "us_per_launch": t, "achieved": 2.0 * M * In * G2 / t / 1e6, "unit": "TFLOP/s",
        "frac": 2.0 * M * In * G2 / t / 1e6 / pk["bf16_tflops"]}
    roof["same_engine_other_shapes"] = others
    del dpre16, wb16, xb16, dx, dw
    # the same contraction on the TF32 engine (operands fp32 in HBM), for reference
    A32 = torch.randn(M, K, device=dev)
    W32 = torch.randn(N, K, device=dev) * 0.05
    us32 = _time_launches(torch, lambda i: ops.gemm(A32, K, 0, W32, K, 1, C[i % nbuf], N, M, N, K, bias=bias), 8)
    roof["tf32_engine_same_shape"] = {"kernel": "tc::gemm_tf32_kernel<0,0>", "us_per_launch": us32,
                                      "achieved": flop / (us32 * 1e-6) / 1e12, "unit": "TFLOP/s"}
    del A, C, A32, W32
    torch.cuda.empty_cache()

    # ---- fused NIG head + loss (two phases) at 2^22 samples x 3 dims: 192 B/sample algorithmic traffic
    n = 1 << 22
    ev = [torch.randn(n, 3, 4, device=dev) for _ in range(2)]
    tg = [torch.tanh(torch.randn(n, 3, device=dev)) for _ in range(2)]

    def nig_launch(i):
        ops.nig_loss_raw(ev[i % 2], None, tg[i % 2], want_nig=True, want_grad=True)

    us_n = _time_launches(torch, nig_launch, 10, warm=3)
    nbytes = 192.0 * n
    roof["nig_head_loss"] = {"kernel": "deer::nig_loss_stats_kernel + nig_loss_finish_kernel (B=2^22, 3 dims, train)",
                             "bound": "hbm", "achieved": nbytes / (us_n * 1e-6) / 1e9, "peak": pk["hbm_gbs"],
                             "unit": "GB/s", "frac": nbytes / (us_n * 1e-6) / 1e9 / pk["hbm_gbs"],
                             "us_per_call": us_n, "algorithmic_bytes": nbytes,
                             "traffic": NCU_TRAFFIC.get("nig_stats_plus_finish"), "traffic_source": NCU_TRAFFIC_SOURCE}
    del ev, tg
    torch.cuda.empty_cache()
    # the same kernel pair at 2^20 samples: the whole call still moves 201 MB (> 126 MB L2), but the 63 MB of OPERANDS stay
    # in L2 between the two passes (evict_last loads in pass 1), so HBM sees every algorithmic byte once
    n2 = 1 << 20
    ev = [torch.randn(n2, 3, 4, device=dev) for _ in range(4)]
    tg = [torch.tanh(torch.randn(n2, 3, device=dev)) for _ in range(4)]
    us_n2 = _time_launches(torch, lambda i: ops.nig_loss_raw(ev[i % 4], None, tg[i % 4], want_nig=True, want_grad=True),
                           12, warm=3)
    roof["nig_head_loss_l2_resident_operands"] = {
        "kernel": "deer::nig_loss_stats_kernel + nig_loss_finish_kernel (B=2^20, 3 dims, train; 4 rotating input sets)",
        "bound": "hbm", "achieved": 192.0 * n2 / (us_n2 * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
        "frac": 192.0 * n2 / (us_n2 * 1e-6) / 1e9 / pk["hbm_gbs"], "us_per_call": us_n2,
        "algorithmic_bytes": 192.0 * n2}
    del ev, tg
    torch.cuda.empty_cache()

    # ---- persistent LSTM recurrence (one layer, both directions), latency-bound
    from deer_b200._lib import call, ptr
    Bp = (B + 31) // 32 * 32
    pre = torch.randn(T, B, 2, 4 * H, device=dev).half()          # FP16 pre-activations, as in the step
    w = [torch.randn(4 * H, H, device=dev) * 0.05 for _ in range(2)]
    h = torch.empty(T, B, 2 * H, device=dev)
    hb16 = torch.empty(T, B, 2 * H, device=dev, dtype=torch.bfloat16)
    gact = torch.empty(T * 2 * Bp * 4 * H, device=dev, dtype=torch.float16)          # FP16 kept gates / cell states
    c = torch.empty(T * 2 * Bp * H, device=dev, dtype=torch.float16)
    dh = torch.randn(T, B, 2 * H, device=dev) * 1e-3
    dpre16 = torch.empty(T, B, 2, 4 * H, device=dev, dtype=torch.bfloat16)
    db = torch.zeros(2, 4 * H, device=dev)
    us_f = _time_launches(torch, lambda i: call("deer_lstm_cluster_fwd_pre16", pre.data_ptr(), ptr(w[0]), ptr(w[1]),
                                                ptr(h), ptr(gact), ptr(c), None, hb16.data_ptr(), T, B, H), 5, warm=2)
    us_b = _time_launches(torch, lambda i: call("deer_lstm_cluster_bwd", ptr(gact), ptr(c), ptr(dh), ptr(w[0]), ptr(w[1]),
                                                None, ptr(db), dpre16.data_ptr(), T, B, H), 5, warm=2)
    rflop = 2.0 * B * 2 * 4 * H * H * T
    # algorithmic HBM bytes per (sample, step, direction) [SURVEY 8d / DESIGN 4]: forward reads the FP16 pre-activations
    # (4H x 2 B) and writes h fp32 (H x 4) + its BF16 shadow (H x 2) + the kept gates / cell state (keep_bytes); BPTT
    # reads the kept gates / cell states (c_t and c_{t-1} are one stream) + dh (H x 4) and writes the BF16 dpre (4H x 2)
    keep_b = LSTM_KEEP_BYTES_PER_UNIT * H
    fwd_bytes = (4 * H * 2 + H * 4 + H * 2 + keep_b) * float(B * T * 2)
    bwd_bytes = (keep_b + H * 4 + 4 * H * 2) * float(B * T * 2)
    roof["lstm_recurrence"] = {"kernel": "tc::lstm_fwd_cluster_kernel / lstm_bwd_cluster_kernel (B=256, T=300, H=256, 2 dirs)",
                               "bound": "latency (serial over T)", "fwd_us_per_step": us_f / T, "bwd_us_per_step": us_b / T,
                               "fwd_tflops": rflop / (us_f * 1e-6) / 1e12, "bwd_tflops": rflop / (us_b * 1e-6) / 1e12,
                               "fwd_algorithmic_bytes": fwd_bytes, "bwd_algorithmic_bytes": bwd_bytes,
                               "fwd_hbm": {"achieved": fwd_bytes / (us_f * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                           "frac": fwd_bytes / (us_f * 1e-6) / 1e9 / pk["hbm_gbs"]},
                               "bwd_hbm": {"achieved": bwd_bytes / (us_b * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                           "frac": bwd_bytes / (us_b * 1e-6) / 1e9 / pk["hbm_gbs"]},
                               "traffic": NCU_TRAFFIC.get("lstm_fwd_keep"), "bwd_traffic": NCU_TRAFFIC.get("lstm_bwd"),
                               "traffic_source": NCU_TRAFFIC_SOURCE}
    del pre, h, hb16, gact, c, dh, dpre16
    torch.cuda.empty_cache()

    # ---- attention pooling (audio encoder shape): the HBM-measurable op of SURVEY 8d -- one pass over [B,T,512] fp32
    Bp_, D = INFER_B, 2 * H
    xs = [torch.randn(T, Bp_, D, device=dev) for _ in range(2)]        # time-major, as the LSTM writes it (2 x 629 MB)
    sc = torch.randn(T * Bp_, device=dev)
    outp = torch.empty(Bp_, D, device=dev)
    wts = torch.empty(Bp_, T, device=dev)
    us_p = _time_launches(torch, lambda i: call("deer_attn_pool_fwd", ptr(xs[i % 2]), D, Bp_ * D, ptr(sc), 1, Bp_, None,
                                                ptr(outp), ptr(wts), Bp_, T, D, 0), 8, warm=2)
    pbytes = float(Bp_ * T * D * 4 + 2 * Bp_ * T * 4 + Bp_ * D * 4)
    roof["attn_pool"] = {"kernel": "deer::attn_pool_fwd_kernel (B=1024, T=300, D=512: online softmax + weighted sum, one pass)",
                         "bound": "hbm", "achieved": pbytes / (us_p * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": pbytes / (us_p * 1e-6) / 1e9 / pk["hbm_gbs"], "us_per_launch": us_p,
                         "algorithmic_bytes": pbytes, "traffic": None}
    del xs, sc, outp, wts
    torch.cuda.empty_cache()
    return roof


if __name__ == "__main__":
    main()
