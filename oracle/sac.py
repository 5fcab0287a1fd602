"""Oracle: the SAC and "TQC" off-policy updates, NumPy float32.

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.

Restates on explicit batches and explicit ``rsample`` noise:
  * ``SACActorModel`` src/model.py:86-141 -- L x (Linear -> BatchNorm1d (train mode: batch
    statistics, running statistics updated even under ``no_grad``) -> ReLU), ``mean_head``,
    ``log_std_head`` (clamp -20..2), ``x = mean + std * eps``, ``a = tanh(x)``,
    ``log pi = sum(Normal.log_prob(x) - log(1 - a^2 + 1e-8))``
  * ``SACAgent``  src/agent.py:388-770: ``critic_update`` :548-639 (target
    ``min(Q1_t, Q2_t) - 0.2 log pi'`` -- the entropy coefficient is the literal 0.2, the learned
    alpha never enters a loss; MSE; both critics clipped; AdamW), ``actor_update`` :513-530,
    ``alpha_update`` :532-546, ``update`` :659-699 (Polyak only when ``step % gradient_step == 0``)
  * ``TQCAgent``  src/agent.py:773-1171: 5 scalar critics, target = mean of the 3 smallest
    target-critic values per sample (sort over the critic axis, drop the top 2, :971-976) minus
    ``alpha * log pi'``; per-critic MSE / clip / AdamW :987-1011; logged Q is the mean over the
    STEPPED critics :1016-1019; ``actor_update`` :912-934 uses ``alpha.detach()``; Polyak every
    step :1086.
Both share one implementation: an ensemble of ``n`` critics of which the ``n - drop`` smallest
values are averaged (SAC: n = 2, drop = 1, i.e. the minimum).

Pinned by ``tests/golden/sac_*.npz`` / ``tqc_*.npz`` (unmodified reference classes, recorded
``rsample`` draws).
"""
from __future__ import annotations

import math

import numpy as np

from .ddpg import (AdamState, CosineAnnealingLR, F32, clip_grad_norm_, clone_params, grad_norm_python,
                   mlp_backward, mlp_forward)

ADAMW_WD = 0.01
BN_EPS = F32(1e-5)          # nn.BatchNorm1d defaults
BN_MOMENTUM = F32(0.1)
LOG_STD_MIN, LOG_STD_MAX = F32(-20.0), F32(2.0)
LOG_SQRT_2PI = F32(math.log(math.sqrt(2 * math.pi)))


def init_sac_actor(rng, in_dim, hidden, act_dim, layers, head_scale=1.0, log_std_bias=0.01):
    """Xavier-uniform Linear weights, bias 0.01 (src/model.py:143-146); BatchNorm affine 1 / 0,
    running mean 0 / var 1 (torch defaults).

    ``head_scale`` / ``log_std_bias`` shrink the two output heads for PARITY FIXTURES: the
    reference's ``log(1 - tanh(x)^2 + 1e-8)`` loses all significance once |x| > ~6 (the fp32
    action is 1 ulp from +-1, so a 1-ulp difference between two tanh implementations moves the
    log-probability by O(1)); the golden cases therefore keep |x| < ~3, where the formula is
    well conditioned and rel 1e-5 is meaningful.  Returns the parameter list in
    ``SACActorModel.parameters()`` order as [tensor, tensor] pairs --
    [W_l, b_l], [bn_weight_l, bn_bias_l] per hidden layer, then [W_mean, b_mean],
    [W_logstd, b_logstd] -- and the running statistics [[mean_l, var_l], ...]."""
    params, stats = [], []
    d = in_dim
    for _ in range(layers):
        bound = math.sqrt(6.0 / (d + hidden))
        params.append([rng.uniform(-bound, bound, (hidden, d)).astype(F32), np.full(hidden, 0.01, F32)])
        params.append([np.ones(hidden, F32), np.zeros(hidden, F32)])
        stats.append([np.zeros(hidden, F32), np.ones(hidden, F32)])
        d = hidden
    for head in range(2):
        bound = math.sqrt(6.0 / (hidden + act_dim))
        w = (rng.uniform(-bound, bound, (act_dim, hidden)) * head_scale).astype(F32)
        params.append([w, np.full(act_dim, 0.01 if head == 0 else log_std_bias, F32)])
    return params, stats


def actor_sample(params, stats, x, eps, train=True, deterministic=False):
    """SACActorModel.sample (src/model.py:125-141).  Returns (action, log_prob [B,1], cache)."""
    L = (len(params) - 2) // 2
    h = np.asarray(x, F32)
    cache = {"x": [], "xhat": [], "invstd": [], "h": []}
    for l in range(L):
        w, b = params[2 * l]
        g, be = params[2 * l + 1]
        z = (h @ w.T + b).astype(F32)
        cache["x"].append(h)
        if train:
            n = z.shape[0]
            mu = z.mean(axis=0, dtype=F32)
            var = ((z - mu) ** 2).mean(axis=0, dtype=F32)
            rm, rv = stats[l]
            rm[...] = (F32(1) - BN_MOMENTUM) * rm + BN_MOMENTUM * mu
            rv[...] = (F32(1) - BN_MOMENTUM) * rv + BN_MOMENTUM * (var * F32(n / (n - 1.0)))
        else:
            mu, var = stats[l]
        invstd = (F32(1) / np.sqrt(var + BN_EPS)).astype(F32)
        xhat = ((z - mu) * invstd).astype(F32)
        y = (xhat * g + be).astype(F32)
        h = np.maximum(y, F32(0))
        cache["xhat"].append(xhat)
        cache["invstd"].append(invstd)
        cache["h"].append(h)
    (wm, bm), (ws, bs) = params[2 * L], params[2 * L + 1]
    mean = (h @ wm.T + bm).astype(F32)
    raw = (h @ ws.T + bs).astype(F32)
    log_std = np.clip(raw, LOG_STD_MIN, LOG_STD_MAX)
    std = np.exp(log_std).astype(F32)
    if deterministic:
        return np.tanh(mean).astype(F32), None, cache
    xt = (mean + std * eps).astype(F32)
    act = np.tanh(xt).astype(F32)
    var_ = (std * std).astype(F32)
    lp = (-((xt - mean) ** 2) / (F32(2) * var_) - np.log(std) - LOG_SQRT_2PI).astype(F32)
    lp = (lp - np.log(F32(1) - act * act + F32(1e-8))).astype(F32)
    logp = lp.sum(axis=-1, keepdims=True, dtype=F32)
    cache.update(mean=mean, raw=raw, std=std, eps=np.asarray(eps, F32), act=act, feat=h)
    return act, logp, cache


def actor_backward(params, cache, d_act, d_logp):
    """Gradients of sum(d_act * action) + sum(d_logp * log_prob) wrt every actor parameter.
    Analytic form of what autograd computes through rsample: d/dmean of the Normal term cancels,
    d/dlog_std of it is -1."""
    L = (len(params) - 2) // 2
    act, std, eps, raw = cache["act"], cache["std"], cache["eps"], cache["raw"]
    one_m = (F32(1) - act * act).astype(F32)
    gx = (d_act * one_m + d_logp * (F32(2) * act * one_m / (one_m + F32(1e-8)))).astype(F32)
    d_mean = gx
    gate = ((raw >= LOG_STD_MIN) & (raw <= LOG_STD_MAX)).astype(F32)
    d_raw = ((gx * eps * std - d_logp) * gate).astype(F32)
    grads = [[np.zeros_like(a), np.zeros_like(b)] for a, b in params]
    feat = cache["feat"]
    (wm, _), (ws, _) = params[2 * L], params[2 * L + 1]
    grads[2 * L] = [(d_mean.T @ feat).astype(F32), d_mean.sum(0, dtype=F32)]
    grads[2 * L + 1] = [(d_raw.T @ feat).astype(F32), d_raw.sum(0, dtype=F32)]
    dh = (d_mean @ wm + d_raw @ ws).astype(F32)
    for l in range(L - 1, -1, -1):
        w, _ = params[2 * l]
        g, _ = params[2 * l + 1]
        xhat, invstd, h = cache["xhat"][l], cache["invstd"][l], cache["h"][l]
        dy = np.where(h > 0, dh, F32(0)).astype(F32)
        n = F32(dy.shape[0])
        dg = (dy * xhat).sum(0, dtype=F32)
        db = dy.sum(0, dtype=F32)
        dxhat = (dy * g).astype(F32)
        dz = (invstd / n * (n * dxhat - dxhat.sum(0, dtype=F32) - xhat * (dxhat * xhat).sum(0, dtype=F32))).astype(F32)
        grads[2 * l + 1] = [dg, db]
        grads[2 * l] = [(dz.T @ cache["x"][l]).astype(F32), dz.sum(0, dtype=F32)]
        if l > 0:
            dh = (dz @ w).astype(F32)
    return grads


def truncated_mean(q, drop):
    """q: [n, B, 1].  Mean over the n - drop smallest per sample (torch.sort(dim=0), slice,
    mean(dim=0)); returns (value [B,1], weights [n,B,1] = d value / d q)."""
    n = q.shape[0]
    keep = n - drop
    order = np.argsort(q, axis=0, kind="stable")
    srt = np.take_along_axis(q, order, axis=0)
    val = (srt[:keep].sum(axis=0, dtype=F32) / F32(keep)).astype(F32)
    wts = np.zeros_like(q)
    np.put_along_axis(wts, order[:keep], F32(1.0) / F32(keep), axis=0)
    return val, wts


class ScalarAdamW:
    """torch.optim.AdamW on the 1-element ``log_alpha`` (src/agent.py:425, :818)."""

    def __init__(self, lr):
        self.lr, self.m, self.v, self.t = lr, F32(0), F32(0), 0

    def step(self, p, g):
        self.t += 1
        p = F32(p * F32(1.0 - self.lr * ADAMW_WD))
        self.m = F32(self.m + F32(0.1) * (g - self.m))
        self.v = F32(self.v * F32(0.999) + F32(0.001) * g * g)
        bc1 = 1.0 - 0.9 ** self.t
        bc2 = 1.0 - 0.999 ** self.t
        denom = F32(np.sqrt(self.v) / F32(bc2 ** 0.5) + F32(1e-8))
        return F32(p - F32(self.lr / bc1) * (self.m / denom))


class SACOracle:
    """algo = 'sac' | 'tqc'."""
    ENSEMBLE = {"sac": 2, "tqc": 5}      # the reference's critic counts; None: any count (a subclass's own critics)

    def __init__(self, algo, actor, actor_stats, critics, *, act_dim, gamma, tau, grad_clip, actor_lr,
                 critic_lr, alpha_lr, alpha_min_steps, gradient_step, actor_lr_min=None, critic_lr_min=None,
                 ac_scheduler_steps=1, cr_scheduler_steps=1, ac_update_freq=1):
        assert algo in ("sac", "tqc")
        self.algo = algo
        self.actor = clone_params(actor)
        self.actor_stats = clone_params(actor_stats)
        self.critics = [clone_params(c) for c in critics]
        self.target_critics = [clone_params(c) for c in critics]
        self.n = len(critics)
        self.drop = 1 if algo == "sac" else 2
        assert self.ENSEMBLE is None or self.n == self.ENSEMBLE[algo]
        self.actor_opt = AdamState(self.actor, ADAMW_WD)
        self.critic_opts = [AdamState(c, ADAMW_WD) for c in self.critics]
        self.actor_sched = CosineAnnealingLR(actor_lr, ac_scheduler_steps,
                                             actor_lr if actor_lr_min is None else actor_lr_min)
        self.critic_scheds = [CosineAnnealingLR(critic_lr, cr_scheduler_steps,
                                                critic_lr if critic_lr_min is None else critic_lr_min)
                              for _ in critics]
        self.gamma, self.tau, self.grad_clip = gamma, tau, grad_clip
        self.gradient_step, self.ac_update_freq = gradient_step, ac_update_freq
        self.alpha_min_steps = alpha_min_steps
        self.target_entropy = F32(-act_dim * 0.5) if algo == "sac" else F32(-act_dim)
        self.log_alpha = F32(0.0)
        self.alpha = F32(1.0)
        self.alpha_opt = ScalarAdamW(alpha_lr)

    def _coef(self):
        return F32(0.2) if self.algo == "sac" else self.alpha

    def critic_update(self, s, a, r, ns, d, eps, weights=None):
        w = None if weights is None else np.asarray(weights, F32).reshape(-1, 1)   # prioritised replay (:577-596)
        na, nlogp, _ = actor_sample(self.actor, self.actor_stats, ns, eps, train=True)
        tin = np.concatenate([ns, na], -1)
        tq = np.stack([mlp_forward(tc, tin, False)[0] for tc in self.target_critics])
        tqv, _ = truncated_mean(tq, self.drop)
        tqv = (tqv - self._coef() * nlogp).astype(F32)
        y = (r + F32(self.gamma) * (F32(1) - d) * tqv).astype(F32)
        cin = np.concatenate([s, a], -1)
        B = s.shape[0]
        losses, gns, tds, qs = [], [], [], []
        fwd = [mlp_forward(c, cin, False) for c in self.critics]   # graphs built before any step
        for i, c in enumerate(self.critics):
            q, acts = fwd[i] if self.algo == "sac" else mlp_forward(c, cin, False)
            diff = (q - y).astype(F32)
            if w is None:
                losses.append(float(np.mean(diff * diff, dtype=F32)))
                dq = (F32(2) * diff / F32(B)).astype(F32)
            else:
                losses.append(float(np.mean(w * (diff * diff), dtype=F32)))
                dq = (F32(2) * diff * w / F32(B)).astype(F32)
            g, _ = mlp_backward(c, acts, dq, False)
            clip_grad_norm_(g, self.grad_clip)
            gns.append(grad_norm_python(g))
            self.critic_opts[i].step(c, g, self.critic_scheds[i].lr)
            if self.algo == "tqc":
                self.critic_scheds[i].step()
            tds.append(np.abs(q - y))
            qs.append(q)
        if self.algo == "sac":
            for sch in self.critic_scheds:
                sch.step()
        td = np.max(np.stack(tds), axis=0).astype(F32)                      # per sample when prioritised (:620-621)
        if w is None:
            td = float(np.mean(td, dtype=F32))
        self.last_y = y
        if self.algo == "sac":
            qv = float(np.mean(np.concatenate(qs, -1), dtype=F32))
            return losses[0], losses[1], td, qv, gns[0], gns[1]
        qv = float(np.mean(np.stack([mlp_forward(c, cin, False)[0] for c in self.critics]), dtype=F32))
        al, ag = float(np.mean(losses)), float(np.mean(gns))
        return al, al, td, qv, ag, ag

    def actor_update(self, s, eps):
        a, logp, cache = actor_sample(self.actor, self.actor_stats, s, eps, train=True)
        cin = np.concatenate([s, a], -1)
        B = s.shape[0]
        fw = [mlp_forward(c, cin, False) for c in self.critics]
        q = np.stack([f[0] for f in fw])
        qv, wts = truncated_mean(q, self.drop)
        coef = self._coef()
        loss = float(np.mean(coef * logp - qv, dtype=F32))
        d_act = np.zeros_like(a)
        for i, c in enumerate(self.critics):
            dq = (-wts[i] / F32(B)).astype(F32)
            _, d_in = mlp_backward(c, fw[i][1], dq, False, need_input_grad=True)
            d_act += d_in[:, s.shape[1]:]
        d_logp = np.full_like(logp, coef / F32(B))
        grads = actor_backward(self.actor, cache, d_act, d_logp)
        clip_grad_norm_(grads, self.grad_clip)
        gn = grad_norm_python(grads)
        self.actor_opt.step(self.actor, grads, self.actor_sched.lr)
        self.actor_sched.step()
        self.last_actor_grads = grads
        return loss, gn, logp

    def alpha_update(self, logp, step):
        if step <= self.alpha_min_steps:
            return 0.0
        t = (logp + self.target_entropy).astype(F32)
        loss = float(-np.mean(self.log_alpha * t, dtype=F32))
        g = F32(-np.mean(t, dtype=F32))
        self.log_alpha = self.alpha_opt.step(self.log_alpha, g)
        self.alpha = F32(np.exp(self.log_alpha))
        return loss

    def _polyak(self):
        t, omt = F32(self.tau), F32(1 - self.tau)
        for tgt, src in zip(self.target_critics, self.critics):
            for (tw, tb), (w, b) in zip(tgt, src):
                tw[...] = t * w + omt * tw
                tb[...] = t * b + omt * tb

    def update_on_batch(self, step, s, a, r, ns, d, eps_next, eps_cur, weights=None):
        l1, l2, td, qv, g1, g2 = self.critic_update(s, a, r, ns, d, eps_next, weights)
        if self.algo == "tqc" or step % self.gradient_step == 0:
            self._polyak()
        if step % self.ac_update_freq == 0:
            al, ag, logp = self.actor_update(s, eps_cur)
            alpha_loss = self.alpha_update(logp, step)
            return l1, l2, al, td, qv, g1, g2, ag, alpha_loss
        return l1, l2, td, qv, g1, g2


# ---- sync-BN (data parallel): the exchange csrc/sac.cu performs between graph segments, restated ----------------
# The reference is single-GPU: nn.BatchNorm1d (src/model.py:103-111) normalises over the whole batch, so N ranks on B
# rows each must equal one rank on the concatenated N * B rows.  These two functions restate what every rank computes
# from the all-gathered slots (bn_fwd_sync_kernel / bn_bwd_sync_kernel); tests/test_sac_oracle_cpu.py checks them
# against the single-batch formulas of actor_sample / actor_backward above on the concatenated batch.
def sync_bn_merge(means, m2s, rows_per_rank):
    """Chan's parallel variance for equal local batches, ranks merged in order: local (mean_r, M2_r = sum (z - mean_r)^2)
    -> (mean, biased variance) of the concatenated batch."""
    means = [np.asarray(m, F32) for m in means]
    world = len(means)
    msum = means[0].copy()
    for m in means[1:]:
        msum = (msum + m).astype(F32)
    mu = (msum / F32(world)).astype(F32)
    m2 = np.zeros_like(mu)
    for m, q in zip(means, m2s):
        d = (m - mu).astype(F32)
        m2 = (m2 + (np.asarray(q, F32) + F32(rows_per_rank) * d * d)).astype(F32)
    return mu, (m2 / (F32(world) * F32(rows_per_rank))).astype(F32)


def sync_bn_backward(dy, xhat, invstd, gamma, s1_all, s2_all, rows_total):
    """Input gradient of one rank's rows: the column sums (sum dy, sum dy * xhat) are taken over ALL ranks (added in
    rank order) and n is the global row count; dgamma / dbeta stay the rank's local sums (they are averaged with the
    flat gradient afterwards)."""
    s1 = np.asarray(s1_all[0], F32).copy()
    s2 = np.asarray(s2_all[0], F32).copy()
    for a, b in zip(s1_all[1:], s2_all[1:]):
        s1 = (s1 + a).astype(F32)
        s2 = (s2 + b).astype(F32)
    n = F32(rows_total)
    dxhat = (dy * gamma).astype(F32)
    return (invstd / n * (n * dxhat - s1 * gamma - xhat * (s2 * gamma))).astype(F32)
