"""NumPy fp32 reference for TQC with quantile critics (``TQCAgent(n_quantiles=M, top_quantiles_to_drop_per_net=d)``,
csrc/sac.cu quantile_target_kernel / quantile_huber_kernel), built on the unmodified SAC / TQC oracle (oracle/sac.py):
the actor sample and backward, the critic MLPs, the clip, AdamW, Polyak and the alpha update are the oracle's; only
``critic_update`` and ``actor_update`` are restated.

  * target: the n * M atoms of the target critics at (s', a' ~ pi(s')) pooled per sample and sorted ascending, the
    K = n (M - d) smallest kept, y_j = r + gamma (1 - done) (z_(j) - alpha log pi(a'|s'));
  * critic i: loss_i = mean over (b, k, j) of w_b |tau_k - 1{u < 0}| h(u), u = y_j - Z_ik, tau_k = (k + 0.5) / M,
    h the Huber function with kappa 1; its own clip and AdamW step;
  * actor: mean_b(alpha log pi - mean_{i,k} Z_ik(s, pi(s))), no truncation;
  * metrics: the mean of the per-critic losses and gradient norms, td = mean_b max_i |mean_k Z_ik - mean_j y_j|
    (per sample with prioritised weights), Q = mean of all atoms of the stepped critics.
"""
import numpy as np

from oracle.ddpg import F32, clip_grad_norm_, grad_norm_python, mlp_backward, mlp_forward
from oracle.sac import SACOracle, actor_backward, actor_sample


def taus(M):
    return ((np.arange(M, dtype=F32) + F32(0.5)) / F32(M)).astype(F32)


def quantile_target(tq, nlogp, r, d, gamma, coef, drop):
    """tq [n, B, M] target atoms, nlogp / r / d [B, 1] -> y [B, K], K = n (M - drop), ascending per row."""
    n, B, M = tq.shape
    pooled = np.sort(np.asarray(tq, F32).transpose(1, 0, 2).reshape(B, n * M), axis=1)
    z = pooled[:, :n * (M - drop)]
    return (r + F32(gamma) * (F32(1) - d) * (z - coef * nlogp)).astype(F32)


def quantile_huber(z, y, w=None):
    """One critic: atoms z [B, M], targets y [B, K], importance weights w [B, 1] or None ->
    (loss, dZ [B, M], per-row |mean_k z - mean_j y| [B, 1])."""
    B, M = z.shape
    K = y.shape[1]
    u = (y[:, None, :] - z[:, :, None]).astype(F32)                 # [B, M, K]
    tau = taus(M)[None, :, None]
    wt = np.where(u < 0, F32(1) - tau, tau).astype(F32)
    au = np.abs(u)
    h = np.where(au > 1, au - F32(0.5), F32(0.5) * u * u).astype(F32)
    ww = F32(1) if w is None else np.asarray(w, F32).reshape(B, 1, 1)
    loss = float(np.mean(ww * wt * h, dtype=F32))
    g = (ww * wt * np.clip(u, F32(-1), F32(1))).sum(axis=2, dtype=F32)
    dz = (-g / F32(B * M * K)).astype(F32)
    td = np.abs(z.mean(axis=1, keepdims=True, dtype=F32) - y.mean(axis=1, keepdims=True, dtype=F32)).astype(F32)
    return loss, dz, td


class QuantileTQCOracle(SACOracle):
    """SACOracle('tqc', ...) with critics whose last Linear is H -> n_quantiles, as many as the critic list holds."""
    ENSEMBLE = None

    def __init__(self, actor, actor_stats, critics, *, n_quantiles, drop_per_net, **kw):
        super().__init__("tqc", actor, actor_stats, critics, **kw)
        assert all(c[-1][0].shape[0] == n_quantiles for c in critics)
        self.M, self.drop_q = n_quantiles, drop_per_net

    def critic_update(self, s, a, r, ns, d, eps, weights=None):
        w = None if weights is None else np.asarray(weights, F32).reshape(-1, 1)
        na, nlogp, _ = actor_sample(self.actor, self.actor_stats, ns, eps, train=True)
        tin = np.concatenate([ns, na], -1)
        tq = np.stack([mlp_forward(tc, tin, False)[0] for tc in self.target_critics])
        y = quantile_target(tq, nlogp, r, d, self.gamma, self._coef(), self.drop_q)
        cin = np.concatenate([s, a], -1)
        losses, gns, tds = [], [], []
        for i, c in enumerate(self.critics):
            z, acts = mlp_forward(c, cin, False)
            loss, dz, td = quantile_huber(z, y, w)
            g, _ = mlp_backward(c, acts, dz, False)
            clip_grad_norm_(g, self.grad_clip)
            gns.append(grad_norm_python(g))
            self.critic_opts[i].step(c, g, self.critic_scheds[i].lr)
            self.critic_scheds[i].step()
            losses.append(loss)
            tds.append(td)
        td = np.max(np.stack(tds), axis=0).astype(F32)
        if w is None:
            td = float(np.mean(td, dtype=F32))
        self.last_y = y
        qv = float(np.mean(np.stack([mlp_forward(c, cin, False)[0] for c in self.critics]), dtype=F32))
        al, ag = float(np.mean(losses)), float(np.mean(gns))
        return al, al, td, qv, ag, ag

    def actor_update(self, s, eps):
        a, logp, cache = actor_sample(self.actor, self.actor_stats, s, eps, train=True)
        cin = np.concatenate([s, a], -1)
        B = s.shape[0]
        fw = [mlp_forward(c, cin, False) for c in self.critics]
        z = np.stack([f[0] for f in fw])                                  # [n, B, M]
        n, M = z.shape[0], z.shape[2]
        coef = self._coef()
        qmean = z.transpose(1, 0, 2).reshape(B, n * M).mean(axis=1, keepdims=True, dtype=F32)
        loss = float(np.mean(coef * logp - qmean, dtype=F32))
        dz = np.full((B, M), F32(-1.0) / F32(B * n * M), F32)
        d_act = np.zeros_like(a)
        for i, c in enumerate(self.critics):
            _, d_in = mlp_backward(c, fw[i][1], dz, False, need_input_grad=True)
            d_act += d_in[:, s.shape[1]:]
        d_logp = np.full_like(logp, coef / F32(B))
        grads = actor_backward(self.actor, cache, d_act, d_logp)
        clip_grad_norm_(grads, self.grad_clip)
        gn = grad_norm_python(grads)
        self.actor_opt.step(self.actor, grads, self.actor_sched.lr)
        self.actor_sched.step()
        self.last_actor_grads = grads
        return loss, gn, logp
