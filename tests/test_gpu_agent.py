"""GPU: the agent kernels (csrc/rexsim_agent.cu, called through the C ABI of include/rexsim_agent.h) against the numpy oracle
(oracle/agent_oracle.py).  fp32 kernels vs fp64 oracle: 2e-5 on network outputs (O(1) values, K = 200 dot products),
1e-5 relative on filter statistics, 1e-4 relative on the scans (sums of up to 1000 terms)."""
import os

import numpy as np
import pytest
import torch

from oracle import agent_oracle as AO

pytestmark = pytest.mark.gpu
REF_POLICIES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policies")


def _random_weights(rng, O, A, H1=200, H2=100):
    sh = dict(pW1=(O, H1), pb1=(H1,), pW2=(H1, H2), pb2=(H2,), pW3=(H2, A), pb3=(A,), logstd=(A,),
              vW1=(O, H1), vb1=(H1,), vW2=(H1, H2), vb2=(H2,), vW3=(H2, 1), vb3=(1,))
    w = {k: rng.normal(0, 0.15, s).astype(np.float32) for k, s in sh.items()}
    w["logstd"] = rng.uniform(-1.2, -0.5, A).astype(np.float32)
    return w


@pytest.mark.parametrize("O,A,n", [(4, 2, 4096), (16, 4, 1000), (4, 1, 77), (16, 2, 65536), (8, 3, 300), (4, 5, 129)])
def test_perform_on_the_tensor_cores(O, A, n):
    """tensor_cores=True: layer 2 as tcgen05.mma kind::tf32 (operands rounded to 11 significant bits, fp32 accumulation in
    TMEM).  Against the fp64 oracle and against the fp32 kernel on the same inputs: mean (after tanh) and value within 5e-3
    (measured worst case over 65 536 x 16-input samples with activations up to +-5: 2.8e-3; 7e-4 on the 4-input networks; a K = 200
    dot product of O(1) terms at 2^-11 relative operand error), sampling noise identical (it does not pass through the GEMM)."""
    from rex_gym_b200.agents import ForwardGaussianPolicy
    rng = np.random.default_rng(O * 100 + A + 7)
    w = _random_weights(rng, O, A)
    f = AO.StreamingNormalize((O,), True, True, 5)
    f.update(rng.normal(0.3, 1.7, (5000, O)))
    obs = (rng.normal(0.3, 3.0, (n, O))).astype(np.float32)
    x = torch.from_numpy(obs).cuda()
    outs = {}
    for tcore in (False, True):
        net = ForwardGaussianPolicy(O, A, tensor_cores=tcore)
        net.set_weights(w)
        net.set_filters(f.count, f.mean, f.var_sum, 0, 0.0, 0.0)
        outs[tcore] = {k: t.cpu().numpy() for k, t in net.perform(x, training=True, seed=3, step=2, env_offset=10).items()}
        outs[tcore]["det"] = net.perform(x, training=False)["action"].cpu().numpy()
        net.close()
    sub = slice(0, min(n, 1024))
    _, m, _, v = AO.perform(w, f, obs[sub], False)
    g, r = outs[True], outs[False]
    em, ev = np.abs(g["mean"][sub] - m).max(), np.abs(g["value"][sub] - v).max()
    print("tf32 perform vs oracle: mean %.2e value %.2e; vs fp32 kernel: mean %.2e value %.2e" % (
        em, ev, np.abs(g["mean"] - r["mean"]).max(), np.abs(g["value"] - r["value"]).max()))
    assert em < 5e-3 and ev < 5e-3
    assert np.abs(g["mean"] - r["mean"]).max() < 5e-3 and np.abs(g["value"] - r["value"]).max() < 5e-3
    assert np.abs(g["mean"] - r["mean"]).mean() < 3e-4                                        # typical error: 1e-4
    assert np.abs((g["action"] - g["mean"]) - (r["action"] - r["mean"])).max() < 1e-5      # same noise draw on both paths
    assert np.abs(g["det"] - g["mean"]).max() == 0 and np.isfinite(g["logprob"]).all()


@pytest.mark.parametrize("O,A,n", [(4, 2, 4096), (16, 4, 1000), (4, 1, 64), (4, 8, 77), (16, 2, 65536)])
def test_perform_matches_the_oracle(O, A, n):
    from rex_gym_b200.agents import ForwardGaussianPolicy
    rng = np.random.default_rng(O * 100 + A)
    net = ForwardGaussianPolicy(O, A)
    w = _random_weights(rng, O, A)
    net.set_weights(w)
    f = AO.StreamingNormalize((O,), True, True, 5)
    f.update(rng.normal(0.3, 1.7, (5000, O)))
    net.set_filters(f.count, f.mean, f.var_sum, 0, 0.0, 0.0)
    obs = (rng.normal(0.3, 3.0, (n, O))).astype(np.float32)
    obs[0] = 100.0                                                    # clipped at +-5 after normalisation
    x = torch.from_numpy(obs).cuda()
    sub = slice(0, n) if n <= 4096 else np.r_[0:512, n - 512:n]       # the python oracle draws noise per element
    for training in (False, True):
        out = net.perform(x, training=training, seed=99, step=5, env_offset=1000)
        a, m, lp, v = AO.perform(w, f, obs[sub], training, seed=99, step=5, env_offset=1000 if isinstance(sub, slice) else 0)
        g = {k: t.cpu().numpy() for k, t in out.items()}
        np.testing.assert_allclose(g["mean"][sub], m, atol=2e-5)
        np.testing.assert_allclose(g["value"][sub], v, atol=5e-5)
        if isinstance(sub, slice) or not training:
            np.testing.assert_allclose(g["action"][sub], a, atol=5e-5)
            np.testing.assert_allclose(g["logprob"][sub], lp, atol=2e-4)
        else:                                                          # global env ids differ in the tail block: check the head only
            a2, _, lp2, _ = AO.perform(w, f, obs[:512], True, seed=99, step=5, env_offset=1000)
            np.testing.assert_allclose(g["action"][:512], a2, atol=5e-5)
        assert np.isfinite(g["action"]).all()
    # sampling statistics: (action - mean) / exp(logstd) ~ N(0, 1), fresh per step
    o1 = net.perform(x, training=True, seed=1, step=0); a1 = o1["action"].cpu().numpy(); m1 = o1["mean"].cpu().numpy()
    a2 = net.perform(x, training=True, seed=1, step=1)["action"].cpu().numpy()
    z = (a1 - m1) / np.exp(w["logstd"])[None, :]
    if n >= 1000:
        assert abs(z.mean()) < 0.1 and abs(z.std() - 1) < 0.1
    assert np.abs(a1 - a2).max() > 1e-3
    net.close()


def test_experience_updates_both_filters_like_the_reference():
    from rex_gym_b200.agents import ForwardGaussianPolicy
    rng = np.random.default_rng(5)
    O = 16
    net = ForwardGaussianPolicy(O, 4)
    fo, fr = AO.StreamingNormalize((O,), True, True, 5), AO.StreamingNormalize((), False, True, 10)
    for n in (1, 3, 4096, 70000, 257):
        obs = rng.normal(0.5, 2.0, (n, O)).astype(np.float32)
        rew = rng.normal(0.1, 0.3, (n,)).astype(np.float32)
        net.experience(torch.from_numpy(obs).cuda(), torch.from_numpy(rew).cuda())
        fo.update(obs); fr.update(rew)
        g = net.get_filters()
        assert g["observ_count"] == fo.count and g["reward_count"] == fr.count
        np.testing.assert_allclose(g["observ_mean"], fo.mean, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(g["observ_var_sum"], fo.var_sum, rtol=5e-5, atol=1e-5)
        np.testing.assert_allclose(g["reward_mean"], fr.mean, rtol=2e-5, atol=2e-6)
        np.testing.assert_allclose(g["reward_var_sum"], fr.var_sum, rtol=5e-5, atol=1e-5)
    r = torch.from_numpy(rng.normal(0, 50, 1000).astype(np.float32)).cuda()
    np.testing.assert_allclose(net.transform_reward(r).cpu().numpy(), fr.transform(r.cpu().numpy()), rtol=1e-5, atol=1e-6)
    # bit-reproducible: same batches -> same statistics
    net2 = ForwardGaussianPolicy(O, 4)
    rng = np.random.default_rng(5)
    for n in (1, 3, 4096, 70000, 257):
        obs = rng.normal(0.5, 2.0, (n, O)).astype(np.float32); rew = rng.normal(0.1, 0.3, (n,)).astype(np.float32)
        net2.experience(torch.from_numpy(obs).cuda(), torch.from_numpy(rew).cuda())
    g2 = net2.get_filters()
    np.testing.assert_array_equal(g2["observ_var_sum"], net.get_filters()["observ_var_sum"])
    net.close(); net2.close()


def test_scans_match_the_oracle_in_both_layouts():
    from rex_gym_b200.agents import utility
    rng = np.random.default_rng(6)
    E, L, g = 3000, 257, 0.985
    r, v = rng.normal(size=(E, L)).astype(np.float32), rng.normal(size=(E, L)).astype(np.float32)
    length = rng.integers(0, L + 1, E).astype(np.int32)
    want_r, want_a = AO.discounted_return(r, length, g), AO.lambda_advantage(r, v, length, g)
    rt, vt, lt = torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(length).cuda()
    np.testing.assert_allclose(utility.discounted_return(rt, lt, g).cpu().numpy(), want_r, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(utility.lambda_advantage(rt, vt, lt, g).cpu().numpy(), want_a, rtol=1e-4, atol=2e-4)
    # time-major storage viewed as [E][L]: same answer, coalesced reads
    rtm, vtm = rt.t().contiguous().t(), vt.t().contiguous().t()
    assert rtm.stride() == (1, E)
    np.testing.assert_allclose(utility.discounted_return(rtm, lt, g).cpu().numpy(), want_r, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(utility.lambda_advantage(rtm, vtm, lt, g).cpu().numpy(), want_a, rtol=1e-4, atol=2e-4)
    T, n = 64, 5000
    r, v = rng.normal(size=(T, n)).astype(np.float32), rng.normal(size=(T + 1, n)).astype(np.float32)
    done = rng.random((T, n)) < 0.05
    wr, wa = AO.gae_segments(r, v, done, g, 0.95)
    gr, ga = utility.gae_segments(torch.from_numpy(r).cuda(), torch.from_numpy(v).cuda(), torch.from_numpy(done).cuda(), g, 0.95)
    np.testing.assert_allclose(gr.cpu().numpy(), wr, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(ga.cpu().numpy(), wa, rtol=1e-4, atol=2e-4)


def test_rollout_graph_equals_the_step_by_step_loop():
    """simulate(): T control steps of perform -> env.step -> experience captured as one CUDA graph; same buffers as the
    unrolled loop on twin environments, and consistent with stepping the env by hand with the recorded actions."""
    import rex_gym_b200 as R
    from rex_gym_b200.agents import ForwardGaussianPolicy, Rollout
    n, T = 512, 16
    kw = dict(task="walk", num_envs=n, signal_type="ik", normalize=True, auto_reset=True, max_episode_steps=25, target_position=2.0, backwards=False)
    outs = []
    for use_graph in (False, True):
        env = R.BatchedRexEnv(**kw)
        net = ForwardGaussianPolicy(env.obs_dim, env.action_dim, seed=3)
        ro = Rollout(env, net, T, seed=17, training=True, use_graph=use_graph)
        a = {k: v.clone() for k, v in ro.collect().items()}
        b = {k: v.clone() for k, v in ro.collect().items()}               # second window: continues the episodes
        outs.append((a, b, net.get_filters(), net.launch_count + env.launch_count))
        if use_graph:
            hand = R.BatchedRexEnv(**kw)
            o = torch.from_numpy(hand.reset()).cuda()
            for t in range(T):
                np.testing.assert_allclose(a["observ"][t].cpu().numpy(), o.cpu().numpy(), atol=1e-6)
                o2, r2, d2, _ = hand.step(a["action"][t])
                np.testing.assert_allclose(a["reward"][t].cpu().numpy(), r2.cpu().numpy(), atol=1e-6)
                np.testing.assert_array_equal(a["done"][t].cpu().numpy(), d2.cpu().numpy())
                o = o2.clone()
            hand.close()
        ret, adv = ro.returns_and_advantages(0.985, 0.95)
        wr, wa = AO.gae_segments(b["reward"].cpu().numpy(), b["value"].cpu().numpy(), b["done"].cpu().numpy(), 0.985, 0.95)
        np.testing.assert_allclose(ret.cpu().numpy(), wr, rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(adv.cpu().numpy(), wa, rtol=1e-4, atol=2e-4)
        env.close(); net.close()
    (a0, b0, f0, _), (a1, b1, f1, _) = outs
    for k in a0:
        np.testing.assert_array_equal(a0[k].cpu().numpy(), a1[k].cpu().numpy(), err_msg=k)
        np.testing.assert_array_equal(b0[k].cpu().numpy(), b1[k].cpu().numpy(), err_msg=k)
    assert f0["observ_count"] == f1["observ_count"] == 2 * T * n
    np.testing.assert_array_equal(f0["observ_var_sum"], f1["observ_var_sum"])
    assert b0["done"].any()                                              # LimitDuration(25) fired inside the second window
    assert np.abs((a0["action"] - a0["mean"]).cpu().numpy()).max() > 1e-3   # training: sampled actions


def test_shipped_policy_runs_on_the_device():
    from rex_gym_b200.agents import ForwardGaussianPolicy
    net = ForwardGaussianPolicy.from_tf_checkpoint(os.path.join(REF_POLICIES, "gallop", "ol"))
    assert (net.O, net.A) == (16, 4)
    net.close()
