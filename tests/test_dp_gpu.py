"""GPU: the data-parallel update.  Parity rule (SURVEY 8e): N ranks on per-rank batches b_r equal
one rank on concat(b_r) within the fp32 tolerance (the reduction order differs); with world size 1
the four phases reproduce the fused update bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ddpg as OD
from tests.helpers import weights_close
from tests.test_ddpg_gpu import make_config

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make_agent(D, A, H, L, B, seed=3, cls=None):
    from gcrl_b200 import DDPG
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    ag = (cls or DDPG)(D, A, make_config(hidden_dim=H, layer_count=L, batch_size=B, grad_clip=0.5), None, 1, 40)
    rng = np.random.default_rng(seed)
    ag._set_layers(NET_ACTOR, OD.init_mlp(rng, D, H, A, L))
    ag._set_layers(NET_CRITIC, OD.init_mlp(rng, D + A, H, 1, L))
    ag.update_target_network()
    return ag


def rand_batch(rng, B, D, A):
    import torch
    s = rng.standard_normal((B, D)).astype(np.float32)
    ns = (s + 0.1 * rng.standard_normal((B, D))).astype(np.float32)
    a = rng.uniform(-1, 1, (B, A)).astype(np.float32)
    r = -(rng.random((B, 1)) > 0.3).astype(np.float32)
    d = (rng.random((B, 1)) < 0.1).astype(np.float32)
    return tuple(torch.from_numpy(x).cuda() for x in (s, a, r, ns, d))


def test_world1_phases_equal_fused_update_bitwise():
    D, A, H, L, B = 21, 3, 256, 3, 256
    fused, phased = make_agent(D, A, H, L, B), make_agent(D, A, H, L, B)
    phased.enable_data_parallel(allreduce_mean=lambda t: t)          # world of one: identity
    rng = np.random.default_rng(0)
    for step in (39, 40, 41):
        batch = rand_batch(rng, B, D, A)
        i1, i2 = fused.update(step, batch=batch), phased.update(step, batch=batch)
        assert [float(x) for x in i1] == [float(x) for x in i2]
    for n1, n2 in ((fused.actor, phased.actor), (fused.critic, phased.critic),
                   (fused.target_actor, phased.target_actor), (fused.target_critic, phased.target_critic)):
        for (w, b), (w2, b2) in zip(n1.layers(), n2.layers()):
            assert np.array_equal(w, w2) and np.array_equal(b, b2)
    assert phased._dp.calls == 6


def test_two_emulated_ranks_equal_one_rank_on_concatenated_batch():
    """Two agents on one GPU play ranks 0/1 (phases driven in lock step, gradients averaged with
    torch between them -- exactly what the NCCL all-reduce does); a third agent sees concat(b0, b1)."""
    import torch
    from gcrl_b200._lib import check, lib, vp
    from gcrl_b200.agent import NET_ACTOR, NET_CRITIC
    D, A, H, L, B = 22, 3, 128, 3, 192
    ranks = [make_agent(D, A, H, L, B), make_agent(D, A, H, L, B)]
    single = make_agent(D, A, H, L, 2 * B)
    rng = np.random.default_rng(1)
    stream = vp(torch.cuda.current_stream().cuda_stream)
    for step in (39, 40, 41, 42):
        batches = [rand_batch(rng, B, D, A) for _ in ranks]
        flags = ranks[0]._flags(step)
        for phase in range(4):
            for ag, b in zip(ranks, batches):
                check(lib.gcrl_agent_update_phase(ag._h, phase, None, B, None, *(vp(t.data_ptr()) for t in b), None,
                                                  1e-3, 1e-3, flags, stream))
            if phase in (0, 2):
                net = NET_CRITIC if phase == 0 else NET_ACTOR
                g = [ag.grad_tensor(net) for ag in ranks]
                mean = (g[0] + g[1]) / 2
                g[0].copy_(mean)
                g[1].copy_(mean)
        m = [np.array(ag.read_metrics()) for ag in ranks]
        info = single.update(step, batch=tuple(torch.cat([b0, b1]) for b0, b1 in zip(*batches)))
        want = np.array([float(x) for x in info])
        got = (m[0] + m[1]) / 2
        np.testing.assert_allclose(got[[0, 1, 2, 3]], want[[0, 1, 2, 3]], rtol=5e-5, atol=2e-6)   # means of means
        np.testing.assert_allclose(m[0][[4, 5]], want[[4, 5]], rtol=5e-5, atol=2e-6)               # global grad norms
        np.testing.assert_array_equal(m[0][[4, 5]], m[1][[4, 5]])
    for nets in zip(*[(ag.actor, ag.critic, ag.target_actor, ag.target_critic) for ag in ranks + [single]]):
        l0, l1, ls = (n.layers() for n in nets)
        for (w0, b0), (w1, b1), (ws, bs) in zip(l0, l1, ls):
            assert np.array_equal(w0, w1) and np.array_equal(b0, b1)       # replicas stay identical
            assert weights_close(w0, ws, 1e-3, 4) and weights_close(b0, bs, 1e-3, 4)


def test_two_gpu_nccl_run_matches_single_rank():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.path.join(ROOT, "goal-conditioned-rl-framework_b200"))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29517",
                          os.path.join(ROOT, "tests", "dp_worker.py")], env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "DP_OK" in out.stdout
