"""Cost of per-utterance audio and video lengths, measured in one process, alternating the configurations on the same GPU.

    python tools/lengths_bench.py [--steps 40] [--rounds 5] [--out FILE]

Training step (B = 256, audio T = 300, video T = 50, the data-parallel trainer's whole step captured as a CUDA graph,
inputs resident):
  default       -- no lengths (bench.py's workload)
  full          -- audio_lengths = T for every sample (layer 0 through the projection GEMM + saturation pass)
  ragged        -- audio_lengths uniform in [75, 300]
  video_full    -- video_lengths = 50 for every clip
  video_ragged  -- video_lengths uniform in [12, 50]
  both_ragged   -- audio and video lengths ragged as above
Inference (B = 1024, eval forward captured as a CUDA graph): without lengths, with ragged audio / ragged video lengths.
Kernels (CUDA events over 200 launches each, B = 256): at T = 300 attention pooling forward / backward dense vs
length-aware on the ragged lengths, with the bytes each reads; the layer-0 permute + 16-bit cast dense vs length-aware;
the saturation pass on the FP16 pre-activations.  At T = 50, C = 512 (the video encoder): BatchNorm statistics, BN+ReLU
forward and backward, the Conv1d padding pass (forward with the FP16 hi / lo split, backward un-pad) plain vs
length-aware on ragged video lengths, and the input masking copy.
Prints one JSON object (GPU name and power limit included); --out also writes it to FILE."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TRAIN_B, INFER_B, T = 256, 1024, 300
TV, CV, DV = 50, 512, 256          # video frames, video encoder width, frame features


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")]
    except Exception as e:          # the numbers are still reported, marked as missing this context
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40, help="timed replays per configuration and round")
    ap.add_argument("--rounds", type=int, default=5, help="alternation rounds (median reported)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import deer_b200
    from bench import synth_batch
    from deer_b200 import _lib
    from deer_b200.trainer import DEERDataParallelTrainer, capture_forward

    assert torch.cuda.is_available(), "lengths_bench measures on a CUDA device"
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(4321)

    def ragged(B):
        return torch.randint(75, T + 1, (B,), generator=gen, dtype=torch.int32).to(dev)

    def vragged(B):
        return torch.randint(TV // 4, TV + 1, (B,), generator=gen, dtype=torch.int32).to(dev)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    def median(v):
        v = sorted(v)
        return v[len(v) // 2]

    # ------------------------------------------------------------------ training step
    model = deer_b200.SequenceDEERModel(dropout=0.3).to(dev).train()
    trainer = DEERDataParallelTrainer(model, learning_rate=1e-4, weight_decay=1e-5, gradient_clip=1.0)
    base = synth_batch(TRAIN_B, dev, gen)
    batches = {"default": base, "full": dict(base, audio_lengths=torch.full((TRAIN_B,), T, dtype=torch.int32, device=dev)),
               "ragged": dict(base, audio_lengths=ragged(TRAIN_B)),
               "video_full": dict(base, video_lengths=torch.full((TRAIN_B,), TV, dtype=torch.int32, device=dev)),
               "video_ragged": dict(base, video_lengths=vragged(TRAIN_B))}
    batches["both_ragged"] = dict(base, audio_lengths=batches["ragged"]["audio_lengths"],
                                  video_lengths=batches["video_ragged"]["video_lengths"])
    launches, replays = {}, {}
    for b in batches.values():      # the zeroed scratch arena grows over the first steps: count launches once it is settled
        for _ in range(3):
            trainer.train_step(b)
    torch.cuda.synchronize()
    for name, b in batches.items():
        l0 = _lib.launch_count()
        trainer.train_step(b)
        launches[name] = _lib.launch_count() - l0
        replays[name] = trainer.capture(b)
    train_ms = {k: [] for k in batches}
    for _ in range(args.rounds):
        for name in batches:
            for _ in range(3):
                replays[name]()
            train_ms[name].append(timed(replays[name], args.steps))
    torch.cuda.synchronize()

    # ------------------------------------------------------------------ inference B = 1024
    model.eval()
    ib = synth_batch(INFER_B, dev, gen)
    keys = ("audio_features", "video_features", "text_features", "attention_mask", "linguistic_features")
    ilen = ragged(INFER_B)
    ireplay = {"default": capture_forward(model, *[ib[k] for k in keys])[0],
               "ragged": capture_forward(model, *[ib[k] for k in keys], audio_lengths=ilen)[0],
               "video_ragged": capture_forward(model, *[ib[k] for k in keys], video_lengths=vragged(INFER_B))[0]}
    infer_ms = {k: [] for k in ireplay}
    for _ in range(args.rounds):
        for name, fn in ireplay.items():
            fn()
            infer_ms[name].append(timed(fn, args.steps))
    del ib
    torch.cuda.synchronize()

    # ------------------------------------------------------------------ kernels at B = 256, T = 300
    D, H = 512, 256
    B = TRAIN_B
    lens = batches["ragged"]["audio_lengths"]
    x = torch.randn(T, B, D, device=dev)
    s = torch.randn(T * B, device=dev)
    out = torch.empty(B, D, device=dev)
    wts = torch.empty(B, T, device=dev)
    dout = torch.randn(B, D, device=dev)
    dx = torch.empty_like(x)
    ds = torch.empty(T * B, device=dev)
    xs_b, xs_t, ss_b, ss_t = D, B * D, 1, B
    p = lambda t: t.data_ptr()
    st = lambda: torch.cuda.current_stream().cuda_stream
    L = _lib.load()
    kern = {
        "pool_fwd_dense": lambda: L.deer_attn_pool_fwd(p(x), xs_b, xs_t, p(s), ss_b, ss_t, None, p(out), p(wts), B, T, D,
                                                       0, st()),
        "pool_fwd_len": lambda: L.deer_attn_pool_len_fwd(p(x), xs_b, xs_t, p(s), ss_b, ss_t, p(lens), 0, p(out), p(wts),
                                                         B, T, D, st()),
        "pool_bwd_dense": lambda: L.deer_attn_pool_bwd(p(dout), p(x), xs_b, xs_t, p(s), ss_b, ss_t, None, p(wts), p(dx),
                                                       p(ds), B, T, D, 0, 0, st()),
        "pool_bwd_len": lambda: L.deer_attn_pool_len_bwd(p(dout), p(x), xs_b, xs_t, ss_b, ss_t, p(lens), 0, p(wts),
                                                         p(dx), p(ds), B, T, D, st()),
    }
    In, Kp = 84, 88                                      # the audio encoder's layer-0 input and its padded K
    xa = torch.randn(B, T, In, device=dev)
    xa16 = torch.empty(T * B, Kp, device=dev, dtype=torch.float16)
    xab16 = torch.empty(T * B, Kp, device=dev, dtype=torch.bfloat16)
    kern["permute_cast16_dense"] = lambda: L.deer_permute_bt_cast16(p(xa), p(xa16), p(xab16), B, T, In, Kp, st())
    kern["permute_cast16_len"] = lambda: L.deer_permute_bt_cast16_len(p(xa), p(xa16), p(xab16), p(lens), 0, B, T, In,
                                                                      Kp, 0, st())
    pre16 = torch.empty(T, B, 2, 4 * H, device=dev, dtype=torch.float16)
    kern["mask_pre_fp16_ragged"] = lambda: L.deer_lstm_mask_pre(p(pre16), 1, p(lens), 0, T, B, H, st())
    full = batches["full"]["audio_lengths"]
    kern["mask_pre_fp16_full"] = lambda: L.deer_lstm_mask_pre(p(pre16), 1, p(full), 0, T, B, H, st())
    kern_us = {}
    for name, fn in kern.items():
        assert fn() == 0, name
        torch.cuda.synchronize()
        kern_us[name] = round(timed(fn, 200) * 1e3, 2)

    # ------------------------------------------------------------------ video encoder kernels at B = 256, T = 50, C = 512
    vlens = batches["video_ragged"]["video_lengths"]
    M = B * TV
    xv = torch.randn(B, TV, CV, device=dev)
    yv, dyv, dxv = torch.empty_like(xv), torch.randn(B, TV, CV, device=dev), torch.empty_like(xv)
    gam, bet = torch.rand(CV, device=dev) + 0.5, torch.randn(CV, device=dev)
    dgam, dbet = torch.zeros(CV, device=dev), torch.zeros(CV, device=dev)
    stats = torch.empty(2 * CV + 1, device=dev)
    scratch = torch.empty(2, CV, device=dev)
    xp = torch.empty(B * (TV + 1) + 2, CV, device=dev)
    hi, lo = (torch.empty(B * (TV + 1) + 2, CV, device=dev, dtype=torch.float16) for _ in range(2))
    xin, xin_m = torch.randn(B, TV, DV, device=dev), torch.empty(B, TV, DV, device=dev)
    mean, var = stats[:CV], stats[CV:2 * CV]
    vk = {
        "bn_stats_plain": lambda: L.deer_bn_stats(p(xv), p(stats), M, CV, st()),
        "bn_stats_len": lambda: L.deer_bn_stats_len(p(xv), p(stats), p(vlens), 0, B, TV, CV, st()),
        "bn_relu_fwd_plain": lambda: L.deer_bn_relu_fwd(p(xv), p(mean), p(var), p(gam), p(bet), p(yv), M, CV, 1e-5,
                                                        st()),
        "bn_relu_fwd_len": lambda: L.deer_bn_relu_fwd_len(p(xv), p(mean), p(var), p(gam), p(bet), p(yv), p(vlens), 0, B,
                                                          TV, CV, 1e-5, st()),
        "bn_relu_bwd_plain": lambda: L.deer_bn_relu_bwd(p(dyv), p(xv), p(yv), p(mean), p(var), p(gam), p(dxv), p(dgam),
                                                        p(dbet), p(scratch), M, CV, 1e-5, 1, st()),
        "bn_relu_bwd_len": lambda: L.deer_bn_relu_bwd_len(p(dyv), p(xv), p(yv), p(mean), p(var), p(gam), p(dxv),
                                                          p(dgam), p(dbet), p(scratch), p(vlens), 0, B, TV, CV, 1e-5, 1,
                                                          st()),
        "rows_pad_fwd_plain": lambda: L.deer_rows_pad_fused(p(xv), p(xp), p(hi), p(lo), B, TV, CV, 1, 1, 0, 0.0, 0, 0,
                                                            None, st()),
        "rows_pad_fwd_len": lambda: L.deer_rows_pad_fused_len(p(xv), p(xp), p(hi), p(lo), p(vlens), 0, B, TV, CV, 1, 1,
                                                              0, 0.0, 0, 0, None, st()),
        "rows_pad_bwd_plain": lambda: L.deer_rows_pad_fused(p(xp), p(dxv), None, None, B, TV, CV, 1, 1, 1, 0.0, 0, 0,
                                                            None, st()),
        "rows_pad_bwd_len": lambda: L.deer_rows_pad_fused_len(p(xp), p(dxv), None, None, p(vlens), 0, B, TV, CV, 1, 1,
                                                              1, 0.0, 0, 0, None, st()),
        "input_mask_copy_len": lambda: L.deer_rowscale_len(p(xin), p(xin_m), p(vlens), 0, B, TV, DV, st()),
    }
    assert L.deer_bn_stats_len(p(xv), p(stats), p(vlens), 0, B, TV, CV, st()) == 0
    vkern_us = {}
    for name, fn in vk.items():
        assert fn() == 0, name
        torch.cuda.synchronize()
        vkern_us[name] = round(timed(fn, 200) * 1e3, 2)
    vsum = int(vlens.long().sum())
    sum_len = int(lens.long().sum())
    rows_dense, rows_len = T * B, sum_len
    res = {
        "gpu": gpu_info(torch),
        "train_step_ms": {k: round(median(v), 4) for k, v in train_ms.items()},
        "train_step_ms_all_rounds": {k: [round(x_, 4) for x_ in v] for k, v in train_ms.items()},
        "train_launches_per_step": launches,
        "inference_b1024_ms": {k: round(median(v), 4) for k, v in infer_ms.items()},
        "inference_b1024_ms_all_rounds": {k: [round(x_, 4) for x_ in v] for k, v in infer_ms.items()},
        "kernel_us_b256_t300": kern_us,
        "video_kernel_us_b256_t50_c512": vkern_us,
        "video_bytes": {"bn_activation_pass": M * CV * 4, "input_mask_copy_read": B * TV * DV * 4,
                        "input_mask_copy_valid_read": vsum * DV * 4},
        "video_ragged_mean_length_b256": vsum / B,
        "pool_x_bytes_read": {"dense": rows_dense * D * 4, "len": rows_len * D * 4},
        "ragged_mean_length_b256": sum_len / B,
        "mask_pre_padded_rows_b256": rows_dense - rows_len,
        "config": {"train_batch": TRAIN_B, "inference_batch": INFER_B, "T": T, "ragged": "uniform int in [75, 300]",
                   "video_T": TV, "video_ragged": "uniform int in [12, 50]",
                   "steps": args.steps, "rounds": args.rounds, "cuda_graphs": True},
    }
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
