"""Partially labelled batches (`target_mask`) through the fused DEER loss kernels (csrc/nig.cu, kMask), the loss
modules, the models' compute_loss, the data-parallel trainer and the batch pipeline, against the fp64 reference of
tests/target_mask_oracle.py: losses, gradients (exactly 0 at unlabelled entries, whatever their target values), head
outputs, both load paths of the kernels, dimensions without labels, summed statistics of two half-batches, graph replay
with a changing mask, launch counts, the prefetcher and host validation."""
import pytest
import torch

from helpers import assert_close, cosine

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import importlib

    import deer_b200
    from deer_b200 import _lib, ops
    # by the package's own name: a `deer_b200.trainer` import would load second copies of ops / _lib under the alias
    # and rebind the package's attributes for every test module collected after this one
    _data = importlib.import_module(deer_b200.__name__ + ".data")
    _trainer = importlib.import_module(deer_b200.__name__ + ".trainer")
    DevicePrefetcher = _data.DevicePrefetcher
    DEERDataParallelTrainer, shard_batch = _trainer.DEERDataParallelTrainer, _trainer.shard_batch
    from gen_common import det_state_dict, pooled_inputs, seq_inputs
    import target_mask_oracle as TMO

DEV = "cuda"
TOL = 1e-3
DIMS = ("valence", "arousal", "dominance")


def cu(t):
    return t.to(torch.float32).to(DEV)


def problem(B, D, seed, frac=0.3, scale=2.0):
    """Evidence, clean targets, mask (about `frac` unlabelled) and targets holding NaN / Inf / 1e30 where unlabelled."""
    g = torch.Generator().manual_seed(seed)
    e = torch.randn(B, D, 4, generator=g, dtype=torch.float64) * scale
    e[:, :, 2] = e[:, :, 2].clamp(min=-5.0)
    y = torch.tanh(torch.randn(B, D, generator=g, dtype=torch.float64))
    mask = torch.rand(B, D, generator=g) >= frac
    junk = torch.tensor([float("nan"), float("inf"), -float("inf"), 1e30], dtype=torch.float64)
    y_bad = y.clone()
    y_bad[~mask] = junk[torch.arange(int((~mask).sum())) % 4]
    return e, y, mask, y_bad


def oracle(e, y, mask, **kw):
    ed = e.clone().requires_grad_(True)
    ref = TMO.masked_loss_from_evidence(ed, y, mask, **kw)
    if ref["total_loss"].requires_grad:
        ref["total_loss"].backward()
    return ref, (ed.grad if ed.grad is not None else torch.zeros_like(e))


def check_losses(losses, ref, D):
    v = ref["vector"]
    assert torch.isfinite(losses).all()
    for i in range(5 * D + 2):
        got, want = float(losses[i].detach()), float(v[i])
        assert abs(got - want) <= TOL * max(abs(want), 1e-3), (i, got, want)


def check_grad(grad, ref_grad, mask):
    assert torch.isfinite(grad).all()
    m = mask.to(DEV)
    assert torch.equal(grad[~m], torch.zeros_like(grad[~m]))
    assert cosine(grad, ref_grad) > 0.99999
    assert_close(grad, ref_grad, TOL, "gradient")


# ---------------------------------------------------------------------------------------------- kernels vs oracle
@pytest.mark.parametrize("B", [65, 257, 4099])
def test_fused_head_loss_with_mask_vs_oracle(B):
    e, y, mask, y_bad = problem(B, 3, B, scale=3.0)
    ref, rgrad = oracle(e, y, mask)
    ec = cu(e).requires_grad_(True)
    nig_out, losses, counts = ops.fused_head_loss(ec, cu(y_bad), target_mask=mask.to(DEV))
    losses[-1].backward()
    check_losses(losses, ref, 3)
    check_grad(ec.grad, rgrad, mask)
    assert counts.tolist() == [float(n) for n in mask.sum(0).tolist()]
    nig_plain, _ = ops.fused_head_loss(cu(e), cu(y))
    assert torch.equal(nig_out, nig_plain)           # head outputs at every entry, labelled or not


@pytest.mark.parametrize("B", [65, 257, 4099])
def test_multitask_loss_params_with_mask_vs_oracle(B):
    e, y, mask, y_bad = problem(B, 3, B + 1)
    p = TMO.O.nig_from_evidence(e)
    params = [p[k].clone().requires_grad_(True) for k in ("mu", "nu", "alpha", "beta")]
    ref = TMO.masked_multitask_loss(*params, y, mask)
    ref["total_loss"].backward()
    pc = [cu(t.detach()).requires_grad_(True) for t in params]
    losses, counts = ops.multitask_loss(*pc, cu(y_bad), target_mask=mask.to(torch.uint8).to(DEV))
    losses[-1].backward()
    check_losses(losses, ref, 3)
    got = torch.stack([t.grad for t in pc], -1)
    want = torch.stack([t.grad for t in params], -1)
    check_grad(got, want, mask)


def test_all_ones_mask_equals_no_mask():
    e, y, _, _ = problem(4099, 3, 7)
    l0, g0, n0, _ = ops.nig_loss_raw(cu(e), None, cu(y), want_nig=True)
    ones = torch.ones(4099, 3, dtype=torch.bool, device=DEV)
    l1, g1, n1, _ = ops.nig_loss_raw(cu(e), None, cu(y), want_nig=True, target_mask=ones)
    assert_close(l1, l0, 1e-5, "losses")            # statistics are summed with atomics: equal up to summation order
    assert_close(g1, g0, 1e-5, "gradient")
    assert torch.equal(n1, n0)


@pytest.mark.parametrize("B,D", [(300001, 3), (70001, 1), (1001, 2), (1400000, 3)])
def test_pipelined_and_plain_trips_with_mask(B, D):
    """Both load paths (DEER_OPT_NIG_PIPELINE), element pairs, odd tails, D = 1 / 2 / 3; B = 1.4 M, D = 3 is past the
    L2-keep threshold of the first pass (its streaming-load instantiation)."""
    e, y, mask, y_bad = problem(B, D, B + D)
    res = []
    try:
        for pipe in (1, 0):
            _lib.set_option(8, pipe)
            counts = torch.empty(D, device=DEV)
            losses, dE, nig, _ = ops.nig_loss_raw(cu(e), None, cu(y_bad), want_nig=True, target_mask=mask.to(DEV),
                                                  counts=counts)
            torch.cuda.synchronize()
            res.append((losses.clone(), dE.clone(), nig.clone(), counts.clone()))
    finally:
        _lib.set_option(8, 1)
    (l1, d1, n1, c1), (l0, d0, n0, c0) = res
    assert_close(l1, l0, 1e-5, "losses")
    assert_close(d1, d0, 1e-5, "gradient")
    assert torch.equal(n1, n0) and torch.equal(c1, c0)
    assert c1.tolist() == [float(n) for n in mask.sum(0).tolist()]
    m = mask.to(DEV)
    assert torch.equal(d1[~m], torch.zeros_like(d1[~m])) and torch.equal(d0[~m], torch.zeros_like(d0[~m]))
    ref = TMO.masked_loss_from_evidence(e, y, mask)
    check_losses(l1, ref, D)


def test_dimension_without_labels_and_empty_mask():
    e, y, mask, y_bad = problem(513, 3, 11)
    mask[:, 1] = False
    y_bad[:, 1] = float("nan")
    ref, rgrad = oracle(e, y, mask)
    ec = cu(e).requires_grad_(True)
    _, losses, counts = ops.fused_head_loss(ec, cu(y_bad), target_mask=mask.to(DEV))
    losses[-1].backward()
    check_losses(losses, ref, 3)
    assert torch.equal(losses[5:10].cpu(), torch.zeros(5))
    assert float(counts[1]) == 0.0
    check_grad(ec.grad, rgrad, mask)
    ec = cu(e).requires_grad_(True)
    none = torch.zeros(513, 3, dtype=torch.bool, device=DEV)
    _, losses, counts = ops.fused_head_loss(ec, cu(y_bad), target_mask=none)
    losses[-1].backward()
    assert torch.equal(losses.cpu(), torch.zeros(17)) and torch.equal(counts.cpu(), torch.zeros(3))
    assert torch.equal(ec.grad, torch.zeros_like(ec))


def test_half_batches_with_summed_statistics_equal_the_full_batch():
    """Exact global semantics on one GPU: the statistics of two half-batches summed through stats_hook give the
    full batch's losses, and the two half gradients together are the full gradient."""
    B = 2048
    e, y, mask, y_bad = problem(B, 3, 13)
    E, Y, M = cu(e), cu(y_bad), mask.to(DEV)
    full_l, full_g, _, _ = ops.nig_loss_raw(E, None, Y, target_mask=M)
    n = B // 2
    stats = []
    for r in range(2):
        _, _, _, st = ops.nig_loss_raw(E[r * n:(r + 1) * n].contiguous(), None, Y[r * n:(r + 1) * n].contiguous(),
                                       target_mask=M[r * n:(r + 1) * n], want_grad=False)
        stats.append(st.clone())
    total = stats[0] + stats[1]
    ls, gs = [], []
    for r in range(2):
        l, g, _, _ = ops.nig_loss_raw(E[r * n:(r + 1) * n].contiguous(), None, Y[r * n:(r + 1) * n].contiguous(),
                                      target_mask=M[r * n:(r + 1) * n], stats_hook=lambda s: s.copy_(total))
        ls.append(l.clone())
        gs.append(g.clone())
    assert_close(ls[0], full_l, 1e-5, "losses")
    assert torch.equal(ls[0], ls[1])
    assert_close(torch.cat(gs), full_g, 1e-5, "gradient")


def test_deer_loss_d1_with_mask_vs_oracle():
    """losses.DEERLoss flattens [B,k] predictions into ONE population; the mask is flattened the same way."""
    e, y, mask, y_bad = problem(600, 1, 17)
    p = TMO.O.nig_from_evidence(e)
    params = {k: p[k].clone().requires_grad_(True) for k in ("mu", "nu", "alpha", "beta")}
    ref = TMO.masked_multitask_loss(params["mu"], params["nu"], params["alpha"], params["beta"], y, mask,
                                    cross_dim_weight=0.0)
    ref["total_loss"].backward()
    pc = {k: cu(v.detach()).requires_grad_(True) for k, v in params.items()}
    out = deer_b200.DEERLoss()(pc, cu(y_bad), target_mask=mask.to(DEV))
    out["total_loss"].backward()
    for k in ("total_loss", "nll_loss", "reg_loss", "kl_loss", "ece_loss"):
        got, want = float(out[k]), float(ref[f"d0_{k}"])
        assert abs(got - want) <= TOL * max(abs(want), 1e-3), (k, got, want)
    assert int(out["num_labeled"]) == int(mask.sum()) and out["batch_size"] == 600
    got = torch.cat([pc[k].grad for k in ("mu", "nu", "alpha", "beta")], 1)
    want = torch.cat([params[k].grad for k in ("mu", "nu", "alpha", "beta")], 1)
    check_grad(got, want, mask.expand(-1, 4))


def test_host_validation():
    e, y, mask, _ = problem(64, 3, 19)
    E, Y = cu(e), cu(y)
    for bad in (mask[:32].to(DEV), mask.to(DEV)[:, :2], mask.to(DEV).float(), mask.to(torch.int32).to(DEV), mask):
        with pytest.raises(ops._lib.DeerError):
            ops.fused_head_loss(E, Y, target_mask=bad)
    with pytest.raises(ops._lib.DeerError):
        deer_b200.DEERLoss()({"mu": Y[:, :1], "nu": Y[:, :1].abs() + 1, "alpha": Y[:, :1].abs() + 2,
                              "beta": Y[:, :1].abs() + 1}, Y[:, 0], target_mask=mask.to(DEV))


# ---------------------------------------------------------------------------------------------- models and trainer
def _pooled(seed):
    torch.manual_seed(0)
    model = deer_b200.CompleteDEERModel(deer_b200.ModelConfig(dropout=0.0))
    sd = det_state_dict({k: tuple(v.shape) for k, v in model.state_dict().items()}, seed=seed)
    model.load_state_dict({k: (v.float() if v.is_floating_point() else v) for k, v in sd.items()})
    model = model.to(DEV).train()
    for mod in model.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    return model


def _seq(seed):
    torch.manual_seed(0)
    model = deer_b200.SequenceDEERModel(dropout=0.0)
    sd = det_state_dict({k: tuple(v.shape) for k, v in model.state_dict().items()}, seed=seed)
    model.load_state_dict({k: (v.float() if v.is_floating_point() else v) for k, v in sd.items()})
    return model.to(DEV).train()


def _mask(B, seed, frac=0.3):
    return (torch.rand(B, 3, generator=torch.Generator().manual_seed(seed)) >= frac).to(DEV)


def _pooled_batch(B, seed):
    a, v, t, y = pooled_inputs(B, seed)
    return {"audio_features": cu(a), "video_features": cu(v), "text_features": cu(t), "targets": cu(y)}


def _seq_batch(B, seed):
    keys = ("audio_features", "video_features", "text_features", "attention_mask", "linguistic_features", "targets")
    return {k: cu(t) for k, t in zip(keys, seq_inputs(B, 24, 10, 12, seed=seed))}


@pytest.mark.parametrize("kind", ["pooled", "sequence"])
def test_trainer_step_with_mask_equals_autograd_of_compute_loss(kind):
    model = _pooled(71) if kind == "pooled" else _seq(72)
    model.loss_fn = deer_b200.MultiTaskDEERLoss(task_weights={"valence": 2.0, "arousal": 1.0, "dominance": 0.5},
                                                cross_dim_weight=0.2, reg_weight=0.3, kl_weight=0.05)
    tr = DEERDataParallelTrainer(model)
    B = 40 if kind == "pooled" else 16
    batch = _pooled_batch(B, 73) if kind == "pooled" else _seq_batch(B, 73)
    mask = _mask(B, 74)
    batch["targets"][~mask] = float("nan")
    batch["target_mask"] = mask
    losses = tr.forward_backward(batch)
    g_tr = tr.flat.grads.clone()
    assert torch.isfinite(losses).all() and torch.isfinite(g_tr).all()
    for p in model.parameters():
        p.grad = None
    out = model(batch)
    rep = model.compute_loss(out, batch["targets"], batch["target_mask"])
    assert abs(float(losses[-1]) - float(rep["total_loss"])) <= 1e-6 * abs(float(rep["total_loss"]))
    for i, d in enumerate(DIMS):
        assert int(rep[f"{d}_num_labeled"]) == int(mask[:, i].sum()) and rep[f"{d}_batch_size"] == B
    rep["total_loss"].backward()
    got, want = [], []
    for n, p in model.named_parameters():
        if p.grad is not None:
            o = tr.flat.offsets[tr.flat.names.index(n)]
            got.append(g_tr[o:o + p.numel()])
            want.append(p.grad.flatten())
    assert_close(torch.cat(got), torch.cat(want), 1e-4, "trainer gradient vs autograd of compute_loss")


def test_graph_replay_follows_the_mask_content():
    """The mask is read on the device: a captured step replays with whatever the static mask buffer holds."""
    B = 40
    batch = _pooled_batch(B, 81)
    masks = [_mask(B, 82 + i) for i in range(3)]
    never = ~(masks[0] | masks[1] | masks[2])          # NaN only where no step labels the entry
    batch["targets"][never] = float("nan")
    assert bool(never.any())
    res = []
    for graph in (False, True):
        model = _pooled(83)
        tr = DEERDataParallelTrainer(model)
        b = {k: v.clone() for k, v in batch.items()}
        b["target_mask"] = masks[0].clone()
        if graph:
            replay = tr.capture(b)               # two eager warm-up steps, then the capture
        else:
            for _ in range(2):
                tr.train_step(b)
        out = []
        for m in masks:
            b["target_mask"].copy_(m)
            losses = replay() if graph else tr.train_step(b)
            out.append(losses.clone())
        torch.cuda.synchronize()
        res.append((torch.stack(out), tr.flat.params.clone()))
    (l0, p0), (l1, p1) = res
    assert torch.isfinite(l1).all()
    assert_close(l1, l0, 1e-5, "losses")
    assert_close(p1, p0, 1e-6, "parameters")
    assert float((l0[0] - l0[1]).abs().max()) > 0       # the mask did change between the steps


def test_masked_training_step_launches_as_many_kernels():
    model = _seq(91)
    tr = DEERDataParallelTrainer(model)
    batch = _seq_batch(256, 92)
    counts = []
    for masked in (False, True, False, True):      # the first two steps warm up (lazily created state)
        b = dict(batch)
        if masked:
            b["target_mask"] = _mask(256, 93)
        before = _lib.launch_count()
        tr.train_step(b)
        counts.append(_lib.launch_count() - before)
    torch.cuda.synchronize()
    assert counts[2] == counts[3], counts


def test_nan_targets_with_mask_train_finite():
    model = _pooled(95)
    tr = DEERDataParallelTrainer(model, learning_rate=1e-3)
    for s in range(4):
        b = _pooled_batch(32, 96 + s)
        b["targets"][torch.rand(32, 3, generator=torch.Generator().manual_seed(s)) < 0.4] = float("nan")
        b["target_mask"] = ~torch.isnan(b["targets"])
        losses = tr.train_step(b)
    torch.cuda.synchronize()
    assert torch.isfinite(losses).all() and torch.isfinite(tr.flat.params).all()


# ---------------------------------------------------------------------------------------------- data path
def test_prefetcher_keeps_bool_mask_and_shard_batch_slices_it():
    host = []
    for s in range(3):
        a, v, t, y = pooled_inputs(8, s)
        m = torch.rand(8, 3, generator=torch.Generator().manual_seed(s)) > 0.5
        host.append({"audio_features": a.float(), "video_features": v.float(), "text_features": t.float(),
                     "targets": y.float(), "target_mask": m})
    seen = []
    for dev_batch in DevicePrefetcher(host, DEV):
        assert dev_batch["target_mask"].dtype == torch.bool and dev_batch["target_mask"].is_cuda
        seen.append(dev_batch["target_mask"].cpu().clone())
    assert all(torch.equal(s_, h["target_mask"]) for s_, h in zip(seen, host))
    sh = shard_batch({k: v.to(DEV) for k, v in host[0].items()}, 1, 2)
    assert torch.equal(sh["target_mask"].cpu(), host[0]["target_mask"][4:])
    assert sh["target_mask"].dtype == torch.bool
