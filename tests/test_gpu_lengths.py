"""Per-utterance audio lengths on the B200 (nn.LSTM on pack_padded_sequence + attention pooling over each utterance's own
frames): the audio encoder against the fp64 reference of tests/lengths_oracle.py, padding independence (NaN / noise in the
padded frames), lengths == T against lengths=None, clamping of device lengths, and the composite model through the
data-parallel trainer, its CUDA-graph replay, the device prefetcher and a B = 1024 inference."""
import pytest
import torch

import deer_b200
import lengths_oracle as LO
from deer_b200 import ops
from deer_b200.data import DevicePrefetcher
from deer_b200.trainer import DEERDataParallelTrainer
from gen_common import det_state_dict, seq_inputs
from helpers import assert_close, cosine, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"
SEQ_KEYS = ("audio_features", "video_features", "text_features", "attention_mask", "linguistic_features", "targets")


def encoder(seed):
    enc = deer_b200.EnhancedAudioEncoder({"hidden_dim": 512, "dropout": 0.0})
    shapes = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
    sd64 = det_state_dict(shapes, seed=seed)
    enc.load_state_dict({k: v.float() for k, v in sd64.items()})
    return enc.to(DEV), sd64


def ragged_lengths(B, T, seed):
    """Uniform in [1, T] with 1, T and lengths on both sides of the 16 / 32-column tile boundaries."""
    g = torch.Generator().manual_seed(seed)
    L = torch.randint(1, T + 1, (B,), generator=g)
    fixed = [1, T, min(T, 16), min(T, 17), min(T, 31), min(T, 33), max(1, T - 1)]
    for i, v in enumerate(fixed[:B]):
        L[(i * 7) % B] = v
    return L


def frames(B, T, seed):
    return torch.randn(B, T, 84, generator=torch.Generator().manual_seed(seed))


def pad_fill(x, lengths, value):
    x = x.clone()
    pad = ~LO.valid_mask(lengths, x.shape[0], x.shape[1])
    if value == "noise":
        x[pad] = 1e3 * torch.randn(int(pad.sum()), x.shape[2], generator=torch.Generator().manual_seed(1))
    else:
        x[pad] = value
    return x


def run(enc, x, lengths, train, x_grad=False, probe_seed=3, host_lengths=False):
    """(output, {param name: grad}, dx) of the encoder on x (CPU) with lengths (None, or moved to the GPU first unless
    host_lengths)."""
    enc.train(train)
    enc.zero_grad(set_to_none=True)
    xs = x.to(DEV).requires_grad_(x_grad)
    lens = lengths.to(DEV) if (lengths is not None and not host_lengths) else lengths
    with torch.set_grad_enabled(train):
        y = enc(xs, lens)
    if not train:
        return y.detach(), None, None
    pr = torch.randn(y.shape, generator=torch.Generator().manual_seed(probe_seed)).to(DEV)
    (y * pr).sum().backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().clone() for n, p in enc.named_parameters()}
    return y.detach(), grads, (xs.grad.detach().clone() if x_grad else None)


STRUCTURAL_ZERO = 1e-4   # attention.2.bias: a bias in front of a softmax has an exactly-zero gradient (round-off only)
# Padded LSTM output rows: o = 2^-60 (the saturated sigmoid) times the recurrence kernels' tanh of a ~0 cell state, whose
# ex2-based form 1 - 2 / (1 + 2^(2x log2e)) leaves up to one fp32 ulp of 1 (2^-23): |h| <= 2^-83 ~ 1.03e-25
PAD_H_BOUND = 2.0 ** -82


def assert_grad_cosine(g, ref, what, tol=0.999):
    if float(ref.abs().max()) < STRUCTURAL_ZERO:
        assert float(g.abs().max()) < STRUCTURAL_ZERO, what
    else:
        c = cosine(g, ref)
        assert c >= tol, (what, c)


def assert_grad_rel(g, ref, tol, what):
    if float(ref.abs().max()) < STRUCTURAL_ZERO:
        assert float(g.abs().max()) < STRUCTURAL_ZERO, what
    else:
        r = rel_l2(g, ref)
        assert r <= tol, (what, r, tol)


def oracle(sd64, x, lengths, probe_seed=3):
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd64.items()}
    xd = x.double().requires_grad_(True)
    y = LO.audio_encoder(xd, sdg, lengths=lengths)
    pr = torch.randn(y.shape, generator=torch.Generator().manual_seed(probe_seed)).double()
    (y * pr).sum().backward()
    return y.detach(), {k: v.grad for k, v in sdg.items()}, xd.grad


@pytest.mark.parametrize("T", [24, 300])
@pytest.mark.parametrize("B", [1, 37, 70, 256])
def test_audio_encoder_lengths_matches_oracle(B, T):
    enc, sd64 = encoder(B + T)
    L = ragged_lengths(B, T, B * T) if B > 1 else torch.tensor([max(1, T // 3)])
    x = frames(B, T, B + 2 * T)
    ref, rgrads, rdx = oracle(sd64, x, L)
    # inference
    y, _, _ = run(enc, x, L, train=False)
    assert_close(y, ref, 1e-3, "eval output")
    # training (dropout 0): the production layer-0 path (batch-major input, no input gradient) ...
    y, grads, _ = run(enc, x, L, train=True)
    assert_close(y, ref, 1e-3, "train output")
    for n, g in grads.items():
        assert_grad_cosine(g, rgrads[n], n)
    # ... and the path of an input that needs a gradient (time-major fp32 copy + zeroing cast)
    y, grads, dx = run(enc, x, L, train=True, x_grad=True)
    assert_close(y, ref, 1e-3, "train output (dx path)")
    for n, g in grads.items():
        assert_grad_cosine(g, rgrads[n], n + " (dx path)")
    assert cosine(dx, rdx) >= 0.999
    pad = ~LO.valid_mask(L, B, T)
    assert float(dx.cpu()[pad].abs().sum()) == 0.0, "dx must be exactly 0 at padded frames"


@pytest.mark.parametrize("B,T", [(37, 24), (256, 300)])
def test_padded_lstm_rows_are_zero(B, T):
    enc, _ = encoder(7)
    L = ragged_lengths(B, T, 11)
    x = pad_fill(frames(B, T, 5), L, float("nan")).to(DEV)
    pad = (~LO.valid_mask(L, B, T)).t().to(DEV)          # [T,B]
    w = [p.detach().requires_grad_(True) for p in enc._layer_weights(0)]   # training: the forward keeps its BF16 shadow
    for grad in (True, False):
        with torch.set_grad_enabled(grad):
            h, h16, hb16 = ops.bilstm_layer(x, *w, emit_f16=True, return_bf16=True, x_batch_major=True,
                                            lengths=L.to(DEV))
        assert torch.isfinite(h).all()
        assert float(h[pad].abs().max()) <= PAD_H_BOUND, (grad, float(h[pad].abs().max()))
        assert float(h16[pad].float().abs().max()) == 0.0, (grad, float(h16[pad].float().abs().max()))
        if grad:
            assert float(hb16[pad].float().abs().max()) <= PAD_H_BOUND, float(hb16[pad].float().abs().max())
    # the encoder's last layer
    enc.eval()
    with torch.no_grad():
        h2 = enc.lstm_forward(x, lengths=L.to(DEV))
    assert float(h2[pad].abs().max()) <= PAD_H_BOUND, float(h2[pad].abs().max())


@pytest.mark.parametrize("B,T", [(70, 24), (256, 300)])
@pytest.mark.parametrize("fill", ["nan", "noise"])
def test_padding_content_does_not_matter(B, T, fill):
    enc, _ = encoder(B)
    L = ragged_lengths(B, T, 3)
    x0 = pad_fill(frames(B, T, 9), L, 0.0)
    xf = pad_fill(x0, L, float("nan") if fill == "nan" else "noise")
    for x_grad in (False, True):
        y0, g0, d0 = run(enc, x0, L, train=True, x_grad=x_grad)
        yn, gn, dn = run(enc, x0, L, train=True, x_grad=x_grad)     # run-to-run noise (atomic bias gradients)
        yf, gf, df = run(enc, xf, L, train=True, x_grad=x_grad)
        assert torch.isfinite(yf).all()
        assert rel_l2(yf, y0) <= 1e-6 + 2 * rel_l2(yn, y0)
        for n in g0:
            assert torch.isfinite(gf[n]).all(), n
            assert_grad_rel(gf[n], g0[n], 1e-5 + 2 * rel_l2(gn[n], g0[n]), n)
        if x_grad:
            assert torch.isfinite(df).all()
            assert rel_l2(df, d0) <= 1e-5 + 2 * rel_l2(dn, d0)
    ye, _, _ = run(enc, xf, L, train=False)
    y0e, _, _ = run(enc, x0, L, train=False)
    assert torch.isfinite(ye).all() and rel_l2(ye, y0e) <= 1e-6


@pytest.mark.parametrize("B,T", [(70, 24), (256, 300)])
def test_full_lengths_equal_no_lengths(B, T):
    """lengths == T for every sample runs layer 0 through the projection GEMM + saturation pass instead of the in-kernel
    projection: the same result up to FP16 operand rounding."""
    enc, _ = encoder(B + 1)
    x = frames(B, T, 4)
    full = torch.full((B,), T, dtype=torch.int32)
    for train in (False, True):
        y0, g0, _ = run(enc, x, None, train)
        y1, g1, _ = run(enc, x, full, train)
        assert_close(y1, y0, 1e-3, f"output, train={train}")
        if train:
            for n in g0:
                assert_grad_cosine(g1[n], g0[n], n, 0.9999)


@pytest.mark.parametrize("dtype", [torch.int32, torch.int64])
def test_length_entries_at_full_length_equal_plain_entries(dtype):
    """The length entries launch the pooling and permute-cast kernels of their plain counterparts: with every length
    equal to T they write the same bits (B = 256, T = 300, the audio encoder's pooling and layer-0 operand shapes)."""
    B, T, D, In, Kp = 256, 300, 512, 84, 88
    g = torch.Generator(device=DEV).manual_seed(12)
    x = torch.randn(T, B, D, device=DEV, generator=g)             # time-major, as the audio encoder pools it
    s = torch.randn(T, B, device=DEV, generator=g)
    dout = torch.randn(B, D, device=DEV, generator=g)
    xs_b, xs_t, ss_b, ss_t = D, B * D, 1, B
    full = torch.full((B,), T, dtype=dtype, device=DEV)
    i64 = int(dtype == torch.int64)
    res = []
    for lens in (None, full):
        out, wts = torch.empty(B, D, device=DEV), torch.empty(B, T, device=DEV)
        dx, ds = torch.empty_like(x), torch.empty_like(s)
        if lens is None:
            ops.call("deer_attn_pool_fwd", ops.ptr(x), xs_b, xs_t, ops.ptr(s), ss_b, ss_t, None, ops.ptr(out),
                     ops.ptr(wts), B, T, D, 0)
            ops.call("deer_attn_pool_bwd", ops.ptr(dout), ops.ptr(x), xs_b, xs_t, ops.ptr(s), ss_b, ss_t, None,
                     ops.ptr(wts), ops.ptr(dx), ops.ptr(ds), B, T, D, 0, 0)
        else:
            ops.call("deer_attn_pool_len_fwd", ops.ptr(x), xs_b, xs_t, ops.ptr(s), ss_b, ss_t, lens.data_ptr(), i64,
                     ops.ptr(out), ops.ptr(wts), B, T, D)
            ops.call("deer_attn_pool_len_bwd", ops.ptr(dout), ops.ptr(x), xs_b, xs_t, ss_b, ss_t, lens.data_ptr(), i64,
                     ops.ptr(wts), ops.ptr(dx), ops.ptr(ds), B, T, D)
        res.append({"out": out, "wts": wts, "dx": dx, "ds": ds})
    xa = torch.randn(B, T, In, device=DEV, generator=g)            # batch-first layer-0 input
    for r, lens in zip(res, (None, full)):
        y16 = torch.empty(T * B, Kp, device=DEV, dtype=torch.float16)
        yb16 = torch.empty(T * B, Kp, device=DEV, dtype=torch.bfloat16)
        if lens is None:
            ops.call("deer_permute_bt_cast16", ops.ptr(xa), y16.data_ptr(), yb16.data_ptr(), B, T, In, Kp)
        else:
            ops.call("deer_permute_bt_cast16_len", ops.ptr(xa), y16.data_ptr(), yb16.data_ptr(), lens.data_ptr(), i64,
                     B, T, In, Kp, 0)
        r.update(y16=y16, yb16=yb16)
    torch.cuda.synchronize()
    for k in res[0]:
        assert torch.equal(res[0][k], res[1][k]), k


def test_device_lengths_are_clamped_and_dtypes_agree():
    B, T = 37, 24
    enc, _ = encoder(2)
    x = frames(B, T, 6)
    L = ragged_lengths(B, T, 8)
    L[3], L[5] = 1, T
    wild = L.clone()
    wild[3], wild[5] = 0, T + 5                            # device lengths are clamped to [1, T]
    y_ref, g_ref, _ = run(enc, x, L.to(torch.int64), train=True)
    for lens in (wild.to(torch.int64), wild.to(torch.int32), L.to(torch.int32)):
        y, g, _ = run(enc, x, lens, train=True)
        assert rel_l2(y, y_ref) <= 1e-5
        for n in g:
            assert_grad_rel(g[n], g_ref[n], 1e-4, n)      # atomically accumulated reductions
    # host lengths: validated, copied
    y, _, _ = run(enc, x, L, train=False, host_lengths=True)
    y_ref_e, _, _ = run(enc, x, L, train=False)
    assert torch.equal(y, y_ref_e)
    with pytest.raises(ops._lib.DeerError):
        run(enc, x, wild, train=False, host_lengths=True)


def test_other_lstm_engines_refuse_lengths():
    enc, _ = encoder(1)
    x = frames(4, 6, 1).to(DEV)
    w = [p.detach() for p in enc._layer_weights(0)]
    ops.set_lstm_engine(ops.ENGINE_SIMT)
    try:
        with pytest.raises(ops._lib.DeerError):
            ops.bilstm_layer(ops.to_time_major(x), *w, lengths=torch.tensor([3, 6, 1, 2], device=DEV))
    finally:
        ops.set_lstm_engine(ops.ENGINE_AUTO)


# ---------------------------------------------------------------------------------------------- composite model
def seq_model(seed):
    torch.manual_seed(0)
    model = deer_b200.SequenceDEERModel(dropout=0.0)
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    sd64 = det_state_dict(shapes, seed=seed)
    model.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in sd64.items()})
    return model.to(DEV), sd64


def seq_batch(B, Ta, seed):
    raw = seq_inputs(B, Ta, 50, 64, seed=seed)
    batch = {k: t.float().to(DEV) for k, t in zip(SEQ_KEYS, raw)}
    L = ragged_lengths(B, Ta, seed)
    L[L < Ta // 4] = Ta // 4            # uniform-ish in [T/4, T] as a corpus would be
    batch["audio_lengths"] = L.to(DEV)
    return raw, batch, L


def test_trainer_step_with_audio_lengths_matches_oracle():
    B, Ta = 256, 300
    model, sd64 = seq_model(5)
    model.train()
    raw, batch, L = seq_batch(B, Ta, 5)
    trainer = DEERDataParallelTrainer(model)
    losses = trainer.forward_backward(batch)
    grads = trainer.flat.grads.clone()
    torch.cuda.synchronize()
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd64.items()}
    _, rloss = LO.sequence_model_loss(*raw[:5], raw[5], sdg, training=True, lengths=L)
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


def test_graph_replayed_step_with_audio_lengths_equals_eager():
    B, Ta = 256, 300
    _, batch, _ = seq_batch(B, Ta, 7)
    res = []
    for auto in (False, False, True):            # two eager runs give the run-to-run noise of the atomic reductions
        model, _ = seq_model(7)
        trainer = DEERDataParallelTrainer(model.train())
        for _ in range(4):                       # auto: 2 eager steps, then capture + replay, replay
            losses = trainer.train_step_auto(batch) if auto else trainer.train_step(batch)
        torch.cuda.synchronize()
        assert torch.isfinite(losses).all()
        res.append((losses.clone(), trainer.flat.params.clone()))
    for i in range(2):
        noise = rel_l2(res[1][i], res[0][i])
        assert rel_l2(res[2][i], res[0][i]) <= 3 * noise + 1e-6, (i, rel_l2(res[2][i], res[0][i]), noise)


def test_prefetcher_stages_audio_lengths_with_its_dtype():
    host = []
    for s in range(3):
        raw = seq_inputs(8, 20, 6, 8, seed=s)
        b = {k: t.float() for k, t in zip(SEQ_KEYS, raw)}
        b["audio_lengths"] = torch.arange(1, 9, dtype=torch.int32) + s
        host.append(b)
    seen = []
    for dev_batch in DevicePrefetcher(host, DEV):
        assert dev_batch["audio_lengths"].dtype == torch.int32 and dev_batch["audio_lengths"].is_cuda
        seen.append(dev_batch["audio_lengths"].cpu().tolist())
    assert seen == [h["audio_lengths"].tolist() for h in host]


def test_inference_b1024_with_audio_lengths_matches_oracle():
    B, Ta = 1024, 300
    model, sd64 = seq_model(9)
    model.eval()
    raw, batch, L = seq_batch(B, Ta, 9)
    with torch.no_grad():
        out = model(batch)
        ref = LO.sequence_model(*raw[:5], sd64, training=False, lengths=L)
    assert_close(out["audio_encoded"], ref["audio_encoded"], 1e-3, "audio_encoded")
    assert_close(out["mu_all"], ref["mu_all"], 1e-3, "mu_all")
