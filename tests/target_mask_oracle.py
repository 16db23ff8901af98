"""fp64 reference of the DEER multitask loss on a partially labelled batch: losses.MultiTaskDEERLoss (losses.py:229-348)
with each dimension's terms taken on that dimension's labelled rows alone.

For dimension d with N_d labelled entries, the five terms are `oracle.deer_oracle.deer_loss` on those rows (means over
N_d, ECE bins holding only labelled entries with the reference's float32-rounded bin weight n_k / N_d), and 0 when
N_d = 0.  u_d is the mean of beta / (alpha - 1 + 1e-8) over the labelled entries, the cross-dimension term averages
(u_i - u_j)^2 over the pairs of dimensions that both have labels (0 with fewer than two), and
total = (sum_d w_d total_d + cross_w * cross) / D.  Unlabelled entries are removed by boolean indexing, so their target
values never enter and autograd gives them an exactly-zero gradient."""
import torch

from oracle import deer_oracle as O

TERMS = ("total_loss", "nll_loss", "reg_loss", "kl_loss", "ece_loss")


def masked_multitask_loss(gamma, nu, alpha, beta, y, mask, reg_weight=0.1, kl_weight=0.01, ece_weight=0.05,
                          cross_dim_weight=0.05, task_weights=None, eps=1e-8):
    """gamma / nu / alpha / beta / y / mask [B,D] (mask: bool, True = labelled).  Returns a dict with per-dimension
    terms `d{i}_{term}`, `d{i}_num_labeled`, `cross_dim_loss`, `total_loss`, and `vector`: the kernels' losses
    [5D+2] layout (per dimension total, nll, reg, kl, ece; cross; total)."""
    mask = mask.bool()
    D = y.shape[1]
    zero = gamma.new_zeros(())
    out, total, ubar = {}, zero, []
    vec = []
    for d in range(D):
        m = mask[:, d]
        n = int(m.sum())
        if n > 0:
            col = lambda t: t[:, d][m]          # noqa: E731  (labelled rows, [N_d])
            r = O.deer_loss(*(col(t).unsqueeze(-1) for t in (gamma, nu, alpha, beta, y)), reg_weight=reg_weight,
                            kl_weight=kl_weight, ece_weight=ece_weight, eps=eps)
            terms = [r[k] for k in TERMS]
            ubar.append((col(beta) / (col(alpha) - 1 + 1e-8)).mean())
        else:
            terms = [zero] * 5
            ubar.append(None)
        w = 1.0 if task_weights is None else task_weights[d]
        total = total + w * terms[0]
        for k, v in zip(TERMS, terms):
            out[f"d{d}_{k}"] = v
        out[f"d{d}_num_labeled"] = n
        vec.extend(terms)
    present = [u for u in ubar if u is not None]
    pairs = [(present[i] - present[j]) ** 2 for i in range(len(present)) for j in range(i + 1, len(present))]
    cross = sum(pairs, zero) / len(pairs) if pairs else zero
    if cross_dim_weight > 0 and D > 1:
        total = total + cross_dim_weight * cross
    out["cross_dim_loss"] = cross
    out["total_loss"] = total / D
    out["vector"] = torch.stack(vec + [cross, out["total_loss"]])
    return out


def masked_loss_from_evidence(e, y, mask, **kw):
    """The same on raw evidence [B,D,4] through the NIG head (deer.py:90-98)."""
    p = O.nig_from_evidence(e)
    return masked_multitask_loss(p["mu"], p["nu"], p["alpha"], p["beta"], y, mask, **kw)
