"""Per-clip video lengths on the B200 (Conv1d taps, BatchNorm statistics and attention pooling over each clip's own
frames): the video encoder against the fp64 reference of tests/video_lengths_oracle.py on both convolution paths (im2col
for B (T + 1) <= 256, sliding window above), padding independence (NaN / noise in the padded frames), lengths == T
against lengths=None, the length entries against their plain counterparts, clamping of device lengths, the fused and the
separate conv dropout, and the composite model through the data-parallel trainer, its CUDA-graph replay, the device
prefetcher and a B = 1024 inference."""
import pytest
import torch

import deer_b200
import lengths_oracle as LO
import video_lengths_oracle as VLO
from deer_b200 import ops
from deer_b200.data import DevicePrefetcher
from deer_b200.trainer import DEERDataParallelTrainer
from gen_common import det_state_dict, seq_inputs
from helpers import assert_close, cosine, rel_l2
from test_gpu_lengths import SEQ_KEYS, assert_grad_cosine, assert_grad_rel, pad_fill, ragged_lengths, seq_model

pytestmark = pytest.mark.gpu
DEV = "cuda"
DIN, D = 256, 512
BNS = ("temporal_cnn.1.", "temporal_cnn.5.")


def encoder(seed, dropout=0.0):
    enc = deer_b200.EnhancedVideoEncoder({"hidden_dim": D, "dropout": dropout, "frame_feature_dim": DIN})
    shapes = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
    sd64 = det_state_dict(shapes, seed=seed)
    enc.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in sd64.items()})
    return enc.to(DEV), sd64


def clip_lengths(B, T, seed):
    """Ragged in [1, T] with 1, 2 and T among them.  A single clip gets 2T/3 frames: BatchNorm over 2 or 3 frames makes
    every gradient upstream of it (nearly) zero in exact arithmetic, and a comparison of those with the reference only
    measures fp32 round-off."""
    L = ragged_lengths(B, T, seed)
    for i, v in enumerate([1, 2, T][:B]):
        L[(i * 5 + 1) % B] = v
    return L if B > 1 else torch.tensor([max(1, 2 * T // 3)])


def frames(B, T, seed):
    return torch.randn(B, T, DIN, generator=torch.Generator().manual_seed(seed))


def running_stats(enc):
    return {bn + k: getattr(enc.temporal_cnn[int(bn.split(".")[1])], k).detach().clone()
            for bn in BNS for k in ("running_mean", "running_var", "num_batches_tracked")}


def run(enc, x, lengths, train, x_grad=False, probe_seed=3, host_lengths=False, fresh_stats=None):
    """(output, {param name: grad}, dx, running statistics after the forward) of the encoder on x (CPU)."""
    if fresh_stats is not None:
        enc.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in fresh_stats.items()})
    enc.train(train)
    enc.zero_grad(set_to_none=True)
    xs = x.to(DEV).requires_grad_(x_grad)
    lens = lengths.to(DEV) if (lengths is not None and not host_lengths) else lengths
    with torch.set_grad_enabled(train):
        y = enc(xs, lens)
    if not train:
        return y.detach(), None, None, None
    pr = torch.randn(y.shape, generator=torch.Generator().manual_seed(probe_seed)).to(DEV)
    (y * pr).sum().backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().clone() for n, p in enc.named_parameters() if p.grad is not None}
    return y.detach(), grads, (xs.grad.detach().clone() if x_grad else None), running_stats(enc)


# Run-to-run noise: the BatchNorm statistics and the reductions of its backward are atomically accumulated, and the
# backward GEMMs take BF16 operands, where an order-dependent last-bit change in dy can move one element's BF16 rounding
# (2^-8): two runs of the same step differ by up to ~1e-4 in the weight gradients and the input gradient.  A comparison
# that should hold up to that noise uses 4x one measured sample of it, or FLOOR_* when that is larger.
FLOOR_OUT, FLOOR_GRAD = 1e-5, 1e-3


def within_noise(got, ref, noisy, floor):
    return rel_l2(got, ref) <= max(floor, 4 * rel_l2(noisy, ref))


def assert_grad_within_noise(got, ref, noisy, what):
    """As within_noise for a parameter gradient; a structural zero (attention.2.bias) is checked as one instead."""
    assert_grad_rel(got, ref, max(FLOOR_GRAD, 4 * rel_l2(noisy, ref)), what)


def oracle(sd64, x, lengths, probe_seed=3):
    """(eval output, training output, {name: grad}, dx, running-statistic updates) of the fp64 reference."""
    ye = VLO.video_encoder(x.double(), sd64, training=False, lengths=lengths)
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd64.items()}
    xd = x.double().requires_grad_(True)
    running = {}
    y = VLO.video_encoder(xd, sdg, training=True, lengths=lengths, running=running)
    pr = torch.randn(y.shape, generator=torch.Generator().manual_seed(probe_seed)).double()
    (y * pr).sum().backward()
    return ye, y.detach(), {k: v.grad for k, v in sdg.items() if v.grad is not None}, xd.grad, running


@pytest.mark.parametrize("T", [8, 50])
@pytest.mark.parametrize("B", [1, 4, 37, 256])
def test_video_encoder_lengths_matches_oracle(B, T):
    """B (T + 1) <= 256 (B = 1, 4 at T = 50; B = 1, 4 at T = 8) runs the im2col convolution, the others the sliding window.
    Below 1024 window rows (B = 37 at T = 8) the convolution's forward runs on TF32 (2^-11 operand rounding, ~3e-4 per
    output element, DESIGN.md 5) rather than split precision, and the batch means in the running statistics carry
    ~1e-4 of it: the running statistics are held to 5e-4 there and to 1e-4 elsewhere."""
    enc, sd64 = encoder(B + T)
    stats_tol = 5e-4 if 256 < B * (T + 1) < 1024 else 1e-4
    L = clip_lengths(B, T, B * T)
    x = pad_fill(frames(B, T, B + 2 * T), L, 0.0)
    ref_e, ref, rgrads, rdx, rrun = oracle(sd64, x, L)
    y, _, _, _ = run(enc, x, L, train=False)
    assert_close(y, ref_e, 1e-3, "eval output")
    pad = ~LO.valid_mask(L, B, T)
    for x_grad in (False, True):
        y, grads, dx, stats = run(enc, x, L, train=True, x_grad=x_grad, fresh_stats=sd64)
        assert_close(y, ref, 1e-3, f"train output (x_grad={x_grad})")
        for n, g in grads.items():
            assert_grad_cosine(g, rgrads[n], n)
        for bn in BNS:
            for k in ("running_mean", "running_var"):
                assert rel_l2(stats[bn + k], rrun[bn + k]) <= stats_tol, (bn + k, rel_l2(stats[bn + k], rrun[bn + k]))
            assert int(stats[bn + "num_batches_tracked"]) == int(sd64[bn + "num_batches_tracked"]) + 1
        if x_grad:
            assert cosine(dx, rdx) >= 0.999
            assert float(dx.cpu()[pad].abs().sum()) == 0.0, "dx must be exactly 0 at padded frames"


@pytest.mark.parametrize("B,T", [(4, 50), (256, 50)])
def test_batchnorm_relu_is_zero_at_padded_rows(B, T):
    """ops.batchnorm_relu with lengths: y exactly 0 at padded rows in training and eval, dx exactly 0 there, NaN padding in
    x changes nothing; the statistics are those of the valid rows (training) and the running update matches nn.BatchNorm1d
    on the packed valid rows."""
    L = clip_lengths(B, T, 5)
    pad = ~LO.valid_mask(L, B, T)
    g = torch.Generator().manual_seed(B)
    x = torch.randn(B, T, D, generator=g) * 2 + 0.5
    gam, bet = torch.rand(D, generator=g) + 0.5, torch.randn(D, generator=g) * 0.1
    dy = torch.randn(B, T, D, generator=g)
    bn = torch.nn.BatchNorm1d(D).double().train()
    bn.weight.data, bn.bias.data = gam.double(), bet.double()
    ref = torch.relu(bn(x[~pad].double()))
    for training in (True, False):
        outs = []
        for fill in (0.0, float("nan")):
            xf = pad_fill(x, L, fill).to(DEV).requires_grad_(True)
            rm, rv, nbt = torch.zeros(D, device=DEV), torch.ones(D, device=DEV), torch.zeros((), dtype=torch.int64,
                                                                                              device=DEV)
            gg, bb = gam.to(DEV).requires_grad_(True), bet.to(DEV).requires_grad_(True)
            y = ops.batchnorm_relu(xf, gg, bb, rm, rv, nbt, training, lengths=L.to(DEV))
            (y * dy.to(DEV)).sum().backward()
            torch.cuda.synchronize()
            assert float(y[pad.to(DEV)].abs().sum()) == 0.0 and float(xf.grad[pad.to(DEV)].abs().sum()) == 0.0
            assert torch.isfinite(y).all() and torch.isfinite(xf.grad).all() and torch.isfinite(gg.grad).all()
            outs.append((y.detach(), xf.grad, gg.grad, bb.grad, rm, rv))
            if training:
                assert_close(y[~pad.to(DEV)], ref, 1e-5, "valid rows vs nn.BatchNorm1d")
                assert rel_l2(rm, bn.running_mean) <= 1e-5 and rel_l2(rv, bn.running_var) <= 1e-5
                assert int(nbt) == 1
        for a, c in zip(outs[0], outs[1]):          # the statistics are atomically accumulated: run-to-run noise
            assert_close(a, c, 1e-5)


@pytest.mark.parametrize("B,T", [(37, 8), (256, 50)])
@pytest.mark.parametrize("fill", ["nan", "noise"])
def test_padding_content_does_not_matter(B, T, fill):
    enc, sd64 = encoder(B)
    L = clip_lengths(B, T, 3)
    x0 = pad_fill(frames(B, T, 9), L, 0.0)
    xf = pad_fill(x0, L, float("nan") if fill == "nan" else "noise")
    for x_grad in (False, True):
        y0, g0, d0, s0 = run(enc, x0, L, train=True, x_grad=x_grad, fresh_stats=sd64)
        yn, gn, dn, sn = run(enc, x0, L, train=True, x_grad=x_grad, fresh_stats=sd64)   # run-to-run noise (atomics)
        yf, gf, df, sf = run(enc, xf, L, train=True, x_grad=x_grad, fresh_stats=sd64)
        assert torch.isfinite(yf).all()
        assert within_noise(yf, y0, yn, FLOOR_OUT)
        for n in g0:
            assert torch.isfinite(gf[n]).all(), n
            assert_grad_within_noise(gf[n], g0[n], gn[n], n)
        for k in s0:
            if s0[k].is_floating_point():
                assert torch.isfinite(sf[k]).all(), k
                assert within_noise(sf[k], s0[k], sn[k], FLOOR_OUT), k
        if x_grad:
            assert torch.isfinite(df).all()
            assert within_noise(df, d0, dn, FLOOR_GRAD)
    ye, _, _, _ = run(enc, xf, L, train=False)
    y0e, _, _, _ = run(enc, x0, L, train=False)
    assert torch.isfinite(ye).all() and rel_l2(ye, y0e) <= 1e-6


@pytest.mark.parametrize("B,T", [(4, 50), (37, 8), (256, 50)])
def test_full_lengths_equal_no_lengths(B, T):
    """lengths == T: the same kernels, length-bounded, plus the input masking copy; equal up to the run-to-run noise of
    the atomically accumulated reductions (BatchNorm statistics, bias and weight gradients)."""
    enc, sd64 = encoder(B + 1)
    x = frames(B, T, 4)
    full = torch.full((B,), T, dtype=torch.int32)
    y0, _, _, _ = run(enc, x, None, train=False)
    y1, _, _, _ = run(enc, x, full, train=False)
    assert torch.equal(y0, y1)
    y0, g0, d0, s0 = run(enc, x, None, train=True, x_grad=True, fresh_stats=sd64)
    yn, gn, dn, sn = run(enc, x, None, train=True, x_grad=True, fresh_stats=sd64)
    y1, g1, d1, s1 = run(enc, x, full, train=True, x_grad=True, fresh_stats=sd64)
    assert within_noise(y1, y0, yn, FLOOR_OUT)
    for n in g0:
        assert_grad_within_noise(g1[n], g0[n], gn[n], n)
    assert within_noise(d1, d0, dn, FLOOR_GRAD)
    for k in s0:
        if s0[k].is_floating_point():
            assert within_noise(s1[k], s0[k], sn[k], FLOOR_OUT), k
        else:
            assert torch.equal(s1[k], s0[k]), k


@pytest.mark.parametrize("dtype", [torch.int32, torch.int64])
def test_length_entries_at_full_length_equal_plain_entries(dtype):
    """The padding pass (both directions, with dropout and the FP16 hi / lo split), BN+ReLU forward and the row copy run
    the kernels of their plain counterparts: with every length equal to T they write the same bits (B = 256, T = 50,
    C = 512, the video encoder's shapes)."""
    B, T, C = 256, 50, 512
    g = torch.Generator(device=DEV).manual_seed(21)
    x = torch.randn(B, T, C, device=DEV, generator=g)
    xp_in = torch.randn(B * (T + 1) + 2, C, device=DEV, generator=g)
    mean, var = torch.randn(C, device=DEV, generator=g), torch.rand(C, device=DEV, generator=g) + 0.5
    gam, bet = torch.randn(C, device=DEV, generator=g), torch.randn(C, device=DEV, generator=g)
    full = torch.full((B,), T, dtype=dtype, device=DEV)
    i64 = int(dtype == torch.int64)
    step = torch.full((1,), 3, dtype=torch.int64, device=DEV)
    P = ops.ptr
    res = []
    for lens in (None, full):
        r = {}
        xp = torch.empty(B * (T + 1) + 2, C, device=DEV)
        hi = torch.empty(B * (T + 1) + 2, C, device=DEV, dtype=torch.float16)
        lo = torch.empty_like(hi)
        dx = torch.empty(B, T, C, device=DEV)
        y = torch.empty(B, T, C, device=DEV)
        rs = torch.empty(B, T, C, device=DEV)
        if lens is None:
            ops.call("deer_rows_pad_fused", P(x), P(xp), hi.data_ptr(), lo.data_ptr(), B, T, C, 1, 1, 0, 0.3, 99, 7,
                     P(step))
            ops.call("deer_rows_pad_fused", P(xp_in), P(dx), None, None, B, T, C, 1, 1, 1, 0.3, 99, 7, P(step))
            ops.call("deer_bn_relu_fwd", P(x), P(mean), P(var), P(gam), P(bet), P(y), B * T, C, 1e-5)
            ops.call("deer_rowscale", P(x), P(torch.ones(B * T, device=DEV)), P(rs), B * T, C)
        else:
            lp = lens.data_ptr()
            ops.call("deer_rows_pad_fused_len", P(x), P(xp), hi.data_ptr(), lo.data_ptr(), lp, i64, B, T, C, 1, 1, 0,
                     0.3, 99, 7, P(step))
            ops.call("deer_rows_pad_fused_len", P(xp_in), P(dx), None, None, lp, i64, B, T, C, 1, 1, 1, 0.3, 99, 7,
                     P(step))
            ops.call("deer_bn_relu_fwd_len", P(x), P(mean), P(var), P(gam), P(bet), P(y), lp, i64, B, T, C, 1e-5)
            ops.call("deer_rowscale_len", P(x), P(rs), lp, i64, B, T, C)
        res.append(dict(xp=xp, hi=hi, lo=lo, dx=dx, y=y, rs=rs))
    torch.cuda.synchronize()
    for k in res[0]:
        assert torch.equal(res[0][k], res[1][k]), k


def test_device_lengths_are_clamped_and_dtypes_agree():
    B, T = 37, 8
    enc, sd64 = encoder(2)
    x = frames(B, T, 6)
    L = clip_lengths(B, T, 8)
    L[3], L[5] = 1, T
    wild = L.clone()
    wild[3], wild[5] = 0, T + 5                            # device lengths are clamped to [1, T]
    y_ref, g_ref, _, s_ref = run(enc, x, L.to(torch.int64), train=True, fresh_stats=sd64)
    for lens in (wild.to(torch.int64), wild.to(torch.int32), L.to(torch.int32)):
        y, g, _, s = run(enc, x, lens, train=True, fresh_stats=sd64)
        assert rel_l2(y, y_ref) <= FLOOR_OUT
        for n in g:
            assert_grad_rel(g[n], g_ref[n], FLOOR_GRAD, n)
        for k in s:
            if s[k].is_floating_point():
                assert rel_l2(s[k], s_ref[k]) <= 1e-5, k
    # host lengths: validated, copied
    y, _, _, _ = run(enc, x, L, train=False, host_lengths=True)
    y_ref_e, _, _, _ = run(enc, x, L, train=False)
    assert torch.equal(y, y_ref_e)
    with pytest.raises(ops._lib.DeerError):
        run(enc, x, wild, train=False, host_lengths=True)


def test_one_frame_batch_runs_the_shortcut_and_ignores_lengths():
    B = 8
    enc, sd64 = encoder(4)
    x = frames(B, 1, 2)
    ones = torch.ones(B, dtype=torch.int64)
    for train in (False, True):
        y0, g0, _, _ = run(enc, x, None, train, fresh_stats=sd64)
        y1, g1, _, s1 = run(enc, x, ones, train, fresh_stats=sd64)
        assert torch.equal(y0, y1)
        if train:
            for n in g0:
                assert_grad_rel(g1[n], g0[n], FLOOR_GRAD, n)
            assert int(s1["temporal_cnn.1.num_batches_tracked"]) == int(sd64["temporal_cnn.1.num_batches_tracked"])
    with pytest.raises(ops._lib.DeerError):
        run(enc, x, torch.full((B,), 2), train=False, host_lengths=True)


@pytest.mark.parametrize("B,T", [(4, 50), (256, 50)])
def test_conv_dropout_fused_and_separate_agree_with_lengths(B, T):
    """Dropout 0.3 in training: the dropout folded into the padding passes and the separate dropout node draw the same masks
    with lengths too; both give dx exactly 0 at padded frames and ignore NaN padding.  (B = 4 is the im2col path, where the
    dropout is always a separate node.)"""
    enc, sd64 = encoder(11, dropout=0.3)
    L = clip_lengths(B, T, 13)
    pad = ~LO.valid_mask(L, B, T)
    x0 = pad_fill(frames(B, T, 14), L, 0.0)
    xn = pad_fill(x0, L, float("nan"))
    res = []
    for fused in (True, False):
        ops.set_conv_dropout_fused(fused)
        try:
            for x in (x0, xn):
                ops.manual_seed(5)
                res.append(run(enc, x, L, train=True, x_grad=True, fresh_stats=sd64))
        finally:
            ops.set_conv_dropout_fused(True)
    y0, g0, d0, s0 = res[0]
    for y, g, d, s in res[1:]:
        assert torch.isfinite(y).all() and torch.isfinite(d).all()
        assert float(d.cpu()[pad].abs().sum()) == 0.0
        assert_close(y, y0, 1e-5, "output")
        assert_close(d, d0, FLOOR_GRAD, "dx")
        for n in g0:
            assert torch.isfinite(g[n]).all(), n
            assert_grad_rel(g[n], g0[n], FLOOR_GRAD, n)


# ---------------------------------------------------------------------------------------------- composite model
def seq_batch(B, seed, audio=False):
    Ta, Tv = 300, 50
    raw = seq_inputs(B, Ta, Tv, 64, seed=seed)
    batch = {k: t.float().to(DEV) for k, t in zip(SEQ_KEYS, raw)}
    Lv = clip_lengths(B, Tv, seed + 1)
    Lv[Lv < Tv // 4] = Tv // 4
    Lv[0], Lv[1] = 1, 2
    batch["video_lengths"] = Lv.to(DEV)
    La = None
    if audio:
        La = ragged_lengths(B, Ta, seed)
        La[La < Ta // 4] = Ta // 4
        batch["audio_lengths"] = La.to(torch.int32).to(DEV)
    return raw, batch, La, Lv


@pytest.mark.parametrize("audio", [False, True])
def test_trainer_step_with_video_lengths_matches_oracle(audio):
    B = 256
    model, sd64 = seq_model(5)
    model.train()
    raw, batch, La, Lv = seq_batch(B, 5, audio)
    trainer = DEERDataParallelTrainer(model)
    losses = trainer.forward_backward(batch)
    grads = trainer.flat.grads.clone()
    torch.cuda.synchronize()
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd64.items()}
    running = {}
    _, rloss = VLO.sequence_model_loss(*raw[:5], raw[5], sdg, training=True, audio_lengths=La, video_lengths=Lv,
                                      running=running)
    rloss["total_loss"].backward()
    lerr = abs(float(losses[-1]) - float(rloss["total_loss"])) / abs(float(rloss["total_loss"]))
    assert lerr <= 1e-3
    got, want = [], []
    for n, o in zip(trainer.flat.names, trainer.flat.offsets):
        og = sdg[n].grad
        if og is not None:
            got.append(grads[o:o + og.numel()].double().cpu())
            want.append(og.flatten())
    assert cosine(torch.cat(got), torch.cat(want)) >= 0.999
    msd = model.state_dict()
    for bn in BNS:
        for k in ("running_mean", "running_var"):
            key = "video_encoder." + bn + k
            assert rel_l2(msd[key], running[key]) <= 1e-4, (key, rel_l2(msd[key], running[key]))


def test_graph_replayed_step_with_video_lengths_equals_eager():
    B = 256
    _, batch, _, _ = seq_batch(B, 7, audio=True)
    res = []
    for auto in (False, False, True):            # two eager runs give the run-to-run noise of the atomic reductions
        model, _ = seq_model(7)
        trainer = DEERDataParallelTrainer(model.train())
        for _ in range(4):                       # auto: 2 eager steps, then capture + replay, replay
            losses = trainer.train_step_auto(batch) if auto else trainer.train_step(batch)
        torch.cuda.synchronize()
        assert torch.isfinite(losses).all()
        rm = model.video_encoder.temporal_cnn[5].running_mean.clone()
        res.append((losses.clone(), trainer.flat.params.clone(), rm))
    for i in range(3):
        noise = rel_l2(res[1][i], res[0][i])
        assert rel_l2(res[2][i], res[0][i]) <= 3 * noise + 1e-6, (i, rel_l2(res[2][i], res[0][i]), noise)


def test_prefetcher_stages_video_lengths_with_its_dtype():
    host = []
    for s in range(3):
        raw = seq_inputs(8, 20, 6, 8, seed=s)
        b = {k: t.float() for k, t in zip(SEQ_KEYS, raw)}
        b["video_lengths"] = torch.arange(1, 9, dtype=torch.int64).clamp(max=6) - (s % 2)
        b["video_lengths"].clamp_(min=1)
        host.append(b)
    seen = []
    for dev_batch in DevicePrefetcher(host, DEV):
        assert dev_batch["video_lengths"].dtype == torch.int64 and dev_batch["video_lengths"].is_cuda
        seen.append(dev_batch["video_lengths"].cpu().tolist())
    assert seen == [h["video_lengths"].tolist() for h in host]


def test_inference_b1024_with_video_lengths_matches_oracle():
    B = 1024
    model, sd64 = seq_model(9)
    model.eval()
    raw, batch, _, Lv = seq_batch(B, 9)
    with torch.no_grad():
        out = model(batch)
        ref = VLO.sequence_model(*raw[:5], sd64, training=False, video_lengths=Lv)
    assert_close(out["video_encoded"], ref["video_encoded"], 1e-3, "video_encoded")
    assert_close(out["mu_all"], ref["mu_all"], 1e-3, "mu_all")
