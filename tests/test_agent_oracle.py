"""CPU: the numpy restatement of the agent glue (oracle/agent_oracle.py) against independent definitions, the TF-checkpoint
reader against every policy the reference ships (tests/golden/policies: the shipped checkpoints cut to the variables the project
restores, tools/gen_policy_golden.py), and the C ABI of include/rexsim_agent.h (symbols only; no GPU here)."""
import os
import re

import numpy as np
import pytest

from oracle import agent_oracle as AO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_POLICIES = os.path.join(ROOT, "tests", "golden", "policies")


def test_agent_abi_exports_every_declared_symbol():
    from rex_gym_b200 import _capi
    L = _capi.load()
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rexsim_agent.h")).read(), flags=re.S)
    names = sorted(set(re.findall(r"\b(rexagent_[a-z0-9_]+)\s*\(", src)))
    assert len(names) == 20 and sorted(_capi.AGENT_EXPORTS) == names
    for n in names:
        assert hasattr(L, n), n
    cfg = _capi.RexAgentConfig(4, 2, 200, 100, 5.0, 10.0)
    import ctypes as C
    assert L.rexagent_policy_floats(C.byref(cfg)) == 21304 and L.rexagent_value_floats(C.byref(cfg)) == 21204    # padded to 4 floats


def test_streaming_normalize_batch_update_equals_definition():
    """normalize.py:73-99: after updates with batches b1..bk, mean and var_sum are those of the concatenated samples."""
    rng = np.random.default_rng(0)
    f = AO.StreamingNormalize((3,), True, True, 5)
    chunks = [rng.normal(1.5, 2.0, (n, 3)) for n in (1, 7, 64, 500)]
    for c in chunks:
        f.update(c)
    allv = np.concatenate(chunks)
    np.testing.assert_allclose(f.mean, allv.mean(0), rtol=1e-12)
    np.testing.assert_allclose(f.var_sum, ((allv - allv.mean(0)) ** 2).sum(0), rtol=1e-10)
    np.testing.assert_allclose(f.std(), np.sqrt(allv.var(0, ddof=1) + 1e-4), rtol=1e-10)
    x = f.transform(allv[:5] * 10)
    assert np.all(np.abs(x) <= 5) and np.any(np.abs(x) == 5)                 # clip
    g = AO.StreamingNormalize((3,), True, True, 5)
    np.testing.assert_array_equal(g.transform(allv[:2]), np.clip(allv[:2], -5, 5))   # count <= 1: no scaling (normalize.py:62-64)


def test_scans_equal_brute_force_sums():
    rng = np.random.default_rng(1)
    E, L, g = 5, 40, 0.985
    r, v = rng.normal(size=(E, L)), rng.normal(size=(E, L))
    length = np.array([40, 1, 17, 0, 33])
    ret, adv = AO.discounted_return(r, length, g), AO.lambda_advantage(r, v, length, g)
    for e in range(E):
        for t in range(L):
            want_r = sum(g ** (k - t) * r[e, k] for k in range(t, L) if k < length[e])
            nv = lambda k: v[e, k + 1] if k + 1 < L else 0.0
            want_a = sum(g ** (k - t) * (r[e, k] + g * nv(k) - v[e, k]) for k in range(t, L) if k < length[e])
            assert abs(ret[e, t] - want_r) < 1e-12 and abs(adv[e, t] - want_a) < 1e-12
    # done-aware time-major form: an episode boundary cuts the sums
    T, n = 12, 3
    r, v = rng.normal(size=(T, n)), rng.normal(size=(T + 1, n))
    done = rng.random((T, n)) < 0.2
    ret, adv = AO.gae_segments(r, v, done, g, 0.9)
    for e in range(n):
        for t in range(T):
            acc, w, k = 0.0, 1.0, t
            while True:
                acc += w * r[k, e]
                if done[k, e]:
                    break
                if k == T - 1:
                    acc += w * g * v[T, e]
                    break
                w *= g; k += 1
            assert abs(ret[t, e] - acc) < 1e-12


def test_network_restatement_equals_a_torch_mlp():
    import torch
    rng = np.random.default_rng(2)
    O, A, H1, H2 = 16, 4, 200, 100
    w = {k: rng.normal(0, 0.1, s).astype(np.float32) for k, s in dict(pW1=(O, H1), pb1=(H1,), pW2=(H1, H2), pb2=(H2,), pW3=(H2, A), pb3=(A,),
                                                                     logstd=(A,), vW1=(O, H1), vb1=(H1,), vW2=(H1, H2), vb2=(H2,), vW3=(H2, 1), vb3=(1,)).items()}
    x = rng.normal(size=(33, O)).astype(np.float32)
    mean, logstd, value = AO.forward_gaussian_policy(w, x)
    t = {k: torch.from_numpy(v).double() for k, v in w.items()}
    xt = torch.from_numpy(x).double()
    h = torch.relu(torch.relu(xt @ t["pW1"] + t["pb1"]) @ t["pW2"] + t["pb2"])
    np.testing.assert_allclose(mean, torch.tanh(h @ t["pW3"] + t["pb3"]).numpy(), atol=1e-12)
    gv = torch.relu(torch.relu(xt @ t["vW1"] + t["vb1"]) @ t["vW2"] + t["vb2"]) @ t["vW3"] + t["vb3"]
    np.testing.assert_allclose(value, gv[:, 0].numpy(), atol=1e-12)
    packed = AO.pack_params(w, O, A, H1, H2)
    back = AO.unpack_params(packed, O, A, H1, H2)
    for k in w:
        np.testing.assert_array_equal(back[k], w[k])


def test_noise_generator_is_the_kernels_generator():
    from rex_gym_b200 import _capi
    L = _capi.load()
    rng = np.random.default_rng(3)
    for _ in range(200):
        s, e, c, k = int(rng.integers(0, 2**63)), int(rng.integers(0, 2**31)), int(rng.integers(0, 2**31)), int(rng.integers(0, 16))
        assert AO.rand_u32(s, e, c, k) == L.rexsim_rand_u32(s, e, c, k)
    z = np.array([AO.normal_noise(7, e, 3, 0) for e in range(4000)])
    assert abs(z.mean()) < 0.06 and abs(z.std() - 1) < 0.05


def test_every_shipped_policy_loads():
    """rex_gym/policies/<task>/<signal>: TF checkpoint-V2 -> ForwardGaussianPolicy layout (200-100 layers, filters)."""
    from rex_gym_b200.agents import tf_checkpoint as tfc
    from rex_gym_b200.agents.networks import read_tf_policy
    want = {"walk/ik": (4, 2), "walk/ol": (4, 8), "gallop/ik": (16, 2), "gallop/ol": (16, 4), "turn/ik": (4, 2), "turn/ol": (4, 2),
            "standup/ol": (4, 1), "poses": (4, 1)}
    for rel, (O, A) in want.items():
        w, filt = read_tf_policy(os.path.join(REF_POLICIES, rel))
        assert w["pW1"].shape == (O, 200) and w["pW2"].shape == (200, 100) and w["pW3"].shape == (100, A) and w["logstd"].shape == (A,)
        assert w["vW3"].shape == (100, 1) and all(np.isfinite(v).all() for v in w.values())
        assert filt[0] >= 1000000 and np.asarray(filt[1]).shape == (O,) and np.all(np.asarray(filt[2]) > 0)
        ents = tfc.list_variables(tfc.latest_checkpoint(os.path.join(REF_POLICIES, rel)))
        assert "global_step" in ents and ents["memory/Variable_1"][1][2] == O
