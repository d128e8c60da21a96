"""CPU restatement of the reference optimizer step (TEST INFRASTRUCTURE - only tests/, smoke() and bench.py's CPU leg
may import this; the product path is clipbert_b200/optim.py + csrc/optim.cu).

Follows src/optimization/adamw.py:40-103 (HuggingFace AdamW with the weight-decay fix) and
torch.nn.utils.clip_grad_norm_ as called at src/tasks/run_video_retrieval.py:477-480. Pinned against the reference's
own class by tests/test_oracle.py, through tests/golden/adamw.pt and tests/golden/reference_live.pt generated from it by
tools/make_golden_adamw.py and tools/make_golden_reference.py.
"""
import math

import torch


def clip_grad_norm(grads, max_norm):
    """Returns (total_norm, clipped grads). torch.nn.utils.clip_grad_norm_: coef = max_norm / (norm + 1e-6), applied
    only when < 1 (norm_type 2)."""
    total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads)).float()
    coef = float(max_norm) / (float(total) + 1e-6)
    if coef < 1.0:
        grads = [g * coef for g in grads]
    return total, grads


def adamw_step(p, g, exp_avg, exp_avg_sq, step, lr, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0, correct_bias=True):
    """One parameter, one step; ``step`` is the 1-based count AFTER the increment (adamw.py:73). Returns (p, m, v)."""
    b1, b2 = betas
    m = exp_avg * b1 + (1.0 - b1) * g                        # adamw.py:76
    v = exp_avg_sq * b2 + (1.0 - b2) * g * g                 # adamw.py:77
    denom = v.sqrt() + eps                                   # adamw.py:78  (eps OUTSIDE the sqrt)
    step_size = lr
    if correct_bias:                                         # adamw.py:81-85
        step_size = step_size * math.sqrt(1.0 - b2 ** step) / (1.0 - b1 ** step)
    p = p - step_size * (m / denom)                          # adamw.py:87
    if weight_decay > 0.0:                                   # adamw.py:98-99: decoupled decay on the UPDATED parameter
        p = p - lr * weight_decay * p
    return p, m, v


def run(params, grads_per_step, groups, max_norm=-1.0):
    """params: list of tensors; groups: list of dict(idx=[param indices], lr, weight_decay, betas, eps, correct_bias);
    grads_per_step: list (steps) of lists (params). Returns the parameter list after every step."""
    ps = [p.clone() for p in params]
    ms = [torch.zeros_like(p) for p in params]
    vs = [torch.zeros_like(p) for p in params]
    traj, norms = [], []
    for t, grads in enumerate(grads_per_step, start=1):
        if max_norm > 0:
            n, grads = clip_grad_norm(grads, max_norm)
            norms.append(n)
        for g in groups:
            for i in g["idx"]:
                ps[i], ms[i], vs[i] = adamw_step(ps[i], grads[i], ms[i], vs[i], t, g["lr"], g.get("betas", (0.9, 0.999)), g.get("eps", 1e-6),
                                                 g.get("weight_decay", 0.0), g.get("correct_bias", True))
        traj.append([p.clone() for p in ps])
    return traj, norms
