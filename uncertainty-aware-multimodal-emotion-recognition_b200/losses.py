"""B200 drop-in for /root/reference/src/utils/losses.py: DEERLoss (:40-226), MultiTaskDEERLoss (:229-348),
CombinedDEERLoss (:500-577) and create_deer_loss (:580).  One fused two-phase CUDA kernel pair computes every term
(NLL, evidence regulariser, KL, ECE bins, cross-dimension consistency) and the analytic gradient; nothing here
synchronises with the host (the reference does 10 host syncs per dimension in the ECE loop, losses.py:217).

Differentiability: `total_loss` carries the gradient; the per-term entries are detached views of the same device
vector (the reference trainer only ever back-propagates total_loss, training.py:216).

Partially labelled batches: every `forward` takes `target_mask` (bool / uint8 CUDA tensor of the targets' shape,
nonzero = labelled).  Each dimension's terms are then the reference's on that dimension's labelled entries alone, the
cross-dimension term averages over the dimensions that have labels, unlabelled target values (NaN, Inf, anything) are
never used and get an exactly-zero gradient, and the output gains `{dim}_num_labeled` (detached 0-d tensors).  Without
a mask nothing changes; in particular a NaN target still makes the loss NaN.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from ._lib import DeerError
from .deer import EVIDENCE_KEY

_TERMS = ("total_loss", "nll_loss", "reg_loss", "kl_loss", "ece_loss")


def _pick(pred, *names):
    for n in names:
        if n in pred and pred[n] is not None:
            return pred[n]
    return None


def _as_col(t: torch.Tensor) -> torch.Tensor:
    return t.unsqueeze(-1) if t.dim() == 1 else t


def _gather(cols: List[torch.Tensor]) -> torch.Tensor:
    """D tensors [B,1] -> contiguous [B,D]; free when they are adjacent column views of one [B,D] buffer."""
    base = cols[0]
    D = len(cols)
    if all(c.dim() == 2 and c.shape[1] == 1 and c.stride(0) == D and c.data_ptr() == base.data_ptr() + 4 * i
           for i, c in enumerate(cols)) and base._base is not None and all(c._base is base._base for c in cols):
        b = base._base
        # (only when the gathered view stays on the autograd tape: a base allocated inside a custom Function's forward
        # -- the [7,B*D] buffer of ops.nig_head -- has no grad_fn, and a view of it would silently detach the head)
        on_tape = (not any(c.requires_grad for c in cols)) or b.requires_grad
        if on_tape and b.dim() >= 2 and b.shape[-1] == D and b.is_contiguous():
            flat = b.reshape(-1, D)
            off = (base.data_ptr() - b.data_ptr()) // (4 * D)
            return flat[off:off + base.shape[0]]
    return torch.cat(cols, dim=1)


class DEERLoss(nn.Module):
    def __init__(self, reg_weight: float = 0.1, kl_weight: float = 0.01, ece_weight: float = 0.05,
                 epsilon: float = 1e-8):
        super().__init__()
        self.reg_weight, self.kl_weight, self.ece_weight, self.epsilon = reg_weight, kl_weight, ece_weight, epsilon

    def forward(self, predictions: Dict[str, torch.Tensor], targets: torch.Tensor,
                target_mask: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        if target_mask is not None and tuple(target_mask.shape) != tuple(targets.shape):
            raise DeerError(f"deer_b200: `target_mask` must have the targets' shape {tuple(targets.shape)}, got "
                            f"{tuple(target_mask.shape)}")
        gamma = _pick(predictions, "gamma", "mu")
        nu = _pick(predictions, "nu", "lambda")
        alpha, beta = predictions.get("alpha"), predictions.get("beta")
        if gamma is None or nu is None or alpha is None or beta is None:
            raise ValueError("Missing required NIG parameters in predictions")
        if targets.dim() == 1 and gamma.dim() == 2:
            targets = targets.unsqueeze(-1)
        elif targets.dim() == 2 and gamma.dim() == 1:
            gamma, nu, alpha, beta = (t.unsqueeze(-1) for t in (gamma, nu, alpha, beta))
        elif targets.dim() == 1:
            gamma, nu, alpha, beta, targets = (t.unsqueeze(-1) for t in (gamma, nu, alpha, beta, targets))
        B = gamma.shape[0]
        # the reference flattens [B,num_dims] into ONE population for the means and the ECE bins (losses.py:150,201)
        # (the mask is flattened the same way)
        flat = [t.reshape(-1, 1) for t in (gamma, nu, alpha, beta)]
        l = ops.multitask_loss(*flat, targets.reshape(-1, 1),
                               weights=(self.reg_weight, self.kl_weight, self.ece_weight, 0.0), eps=self.epsilon,
                               target_mask=None if target_mask is None else target_mask.reshape(-1, 1))
        counts = None
        if target_mask is not None:
            l, counts = l
        out = {"total_loss": l[6]}                      # D=1: [tot,nll,reg,kl,ece, cross, total/1]
        d = l.detach()
        out.update({"nll_loss": d[1], "reg_loss": d[2], "kl_loss": d[3], "ece_loss": d[4], "batch_size": B})
        if counts is not None:
            out["num_labeled"] = counts[0]
        return out


class MultiTaskDEERLoss(nn.Module):
    def __init__(self, emotion_dims: List[str] = ["valence", "arousal", "dominance"],
                 task_weights: Optional[Dict[str, float]] = None, cross_dim_weight: float = 0.05, **deer_loss_kwargs):
        super().__init__()
        self.emotion_dims = list(emotion_dims)
        self.num_dims = len(self.emotion_dims)
        self.cross_dim_weight = cross_dim_weight
        self.task_weights = task_weights or {d: 1.0 for d in self.emotion_dims}
        self.deer_losses = nn.ModuleDict({d: DEERLoss(**deer_loss_kwargs) for d in self.emotion_dims})

    def _weights(self):
        l0 = self.deer_losses[self.emotion_dims[0]]
        return (l0.reg_weight, l0.kl_weight, l0.ece_weight, self.cross_dim_weight), l0.epsilon

    def _task_weight_list(self):
        tw = [float(self.task_weights[d]) for d in self.emotion_dims]
        return None if all(w == 1.0 for w in tw) else tw

    def forward(self, predictions: Dict[str, torch.Tensor], targets: torch.Tensor,
                target_mask: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        w, eps = self._weights()
        D = self.num_dims
        ev = predictions.get(EVIDENCE_KEY)
        if ev is not None and ev.shape[1] == D:
            r = ops.fused_head_loss(ev, targets, w, eps, self._task_weight_list(), target_mask=target_mask)
            l = r[1]
        else:
            cols = {k: [] for k in "gnab"}
            for d in self.emotion_dims:
                g = _pick(predictions, f"{d}_gamma", f"{d}_mu")
                n = _pick(predictions, f"{d}_nu", f"{d}_lambda")
                a, b = predictions[f"{d}_alpha"], predictions[f"{d}_beta"]
                for key, t in zip("gnab", (g, n, a, b)):
                    cols[key].append(_as_col(t))
            r = ops.multitask_loss(_gather(cols["g"]), _gather(cols["n"]), _gather(cols["a"]), _gather(cols["b"]),
                                   targets, w, eps, self._task_weight_list(), target_mask=target_mask)
            l = r if target_mask is None else r[0]
        counts = None if target_mask is None else r[-1]
        det = l.detach()
        out = {}
        for i, d in enumerate(self.emotion_dims):
            for j, term in enumerate(_TERMS):
                out[f"{d}_{term}"] = det[5 * i + j]
            out[f"{d}_batch_size"] = targets.shape[0]
            if counts is not None:
                out[f"{d}_num_labeled"] = counts[i]
        if self.cross_dim_weight > 0 and D > 1:
            out["cross_dim_loss"] = det[5 * D]
        out["total_loss"] = l[5 * D + 1]
        return out


class CombinedDEERLoss(MultiTaskDEERLoss):
    """losses.py:500-577.  On per-dimension prediction dictionaries the reference's extra uncertainty / calibration
    terms read keys (`alpha`,`beta`,`gamma`) that are absent and evaluate to 0.0 (SURVEY.md appendix B#10), so the
    result equals MultiTaskDEERLoss; that behaviour is reproduced."""

    def __init__(self, emotion_dims: List[str] = ["valence", "arousal", "dominance"], deer_weight: float = 1.0,
                 uncertainty_weight: float = 0.1, calibration_weight: float = 0.05, **kwargs):
        super().__init__(emotion_dims=emotion_dims, **kwargs)
        self.deer_weight, self.uncertainty_weight, self.calibration_weight = (deer_weight, uncertainty_weight,
                                                                              calibration_weight)

    def forward(self, predictions, targets, target_mask=None):
        out = super().forward(predictions, targets, target_mask)
        out["deer_loss"] = out["total_loss"]
        if self.deer_weight != 1.0:
            out["total_loss"] = out["total_loss"] * self.deer_weight
        return out


def create_deer_loss(loss_type: str = "multitask", **kwargs) -> nn.Module:
    """losses.py:580 counterpart."""
    if loss_type == "basic":
        return DEERLoss(**kwargs)
    if loss_type == "multitask":
        return MultiTaskDEERLoss(**kwargs)
    if loss_type == "combined":
        return CombinedDEERLoss(**kwargs)
    raise ValueError(f"Unknown loss type: {loss_type}")
