"""Physics parity against REAL PyBullet trajectories.

tests/golden/pybullet_memory_golden.npz holds ALL 25 training episodes per open-loop task (600 control steps of gallop and
walk, the whole 400 of standup), recovered from the PPO EpisodeMemory variables inside the checkpoints the reference ships
(tools/extract_memory_golden.py): policy actions, RangeNormalize'd observations and rewards recorded by the reference's own
RexGymEnv on pybullet==2.8.3.  Open-loop motor commands depend only on the action and the simulation clock, so replaying the
stored actions from the stored reset observation tests pybullet.stepSimulation + the motor model like for like.

Every gallop / walk episode starts from the pristine pose (base at z = 0.21, joints exactly at the task's init pose, zero
velocity: the stored reset observation is exactly that), i.e. a 5 mm free fall onto the feet followed by hopping (gallop) or
stepping (walk).  The replay does NOT diverge chaotically -- the motion is strongly driven -- so the whole 600-step window
(3600 physics sub-steps) is compared.  Measured, fp64 oracle, median over the 25 episodes of the per-episode mean | worst
sample (this round; round 1 in brackets where it was measured):

  gallop-ol joint angles   step 1: 1.5e-5 rad (3.5e-4 before the compound-margin inertias, below)
                           steps 0-20: 1.2e-3 | 2.3e-3 (6e-3)    0-150: 2.3e-3 | 1.6e-2 (4.9e-3 | 2.0e-2)
                           150-300: 4.5e-3 | 3.1e-2    300-450: 4.5e-3 | 3.2e-2    450-600: 4.5e-3 | 2.7e-2
  gallop-ol roll/pitch     0-150: 1.7e-3 | 8.4e-3 (3e-3 | 9e-3)    0-600: 4.2e-3 | 3.7e-2
  walk-ol roll/pitch       0-150: 7.5e-4 | 2.0e-3    0-600: 1.8e-3 | 5.6e-3

  base x (from the recorded rewards: 0 until x > 0.05 m, then x / target): the crossing step agrees with PyBullet's within one
                           control step in 24 of 25 gallop episodes; x(t) over the next ~500 steps within 1-2 % up to the target

The thresholds below are ~1.4x the measured values.  The same file pins the modelling decisions PyBullet's sources left
open or that round 1 had missed (DESIGN.md section 3): combined lateral friction 0.5 (0.48 / 0.52 are already 8 % worse,
0.25 / 1.0 several times), Bullet's 0.04 damping on EVERY link (not only the base: -13 %; 0.2 is worse), the manifold breaking
distance derived the way Bullet derives it (0.81 mm), the effective reach of the toe hull (-0.25 mm: halves the touchdown
error), and the link inertias: Bullet's URDF importer wraps every link's shapes in a btCompoundShape with a 1 mm margin, and the
compound's AABB -- from which the inertia is taken when URDF_USE_INERTIA_FROM_FILE is absent (rex.py:276-287) -- grows by that
margin.  With it the free-fall phase (pure articulated-body dynamics) matches PyBullet 23x better (3.5e-4 -> 1.5e-5 rad after
the first control step) and the first 150 steps 30 % better.  Two more Bullet behaviours are restated because the sources say so, although the gallop / walk recordings cannot
see them (no joint reaches a limit or 100 rad/s there): the +-100 clamp on every generalised velocity and the split-impulse
branch of the joint-limit rows; they decide the standup reset hold (below).
"""
import math
import os

import numpy as np
import pytest

from oracle.oracle import OracleSim

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "pybullet_memory_golden.npz"))
UA, UR = 2 * math.pi + 0.01, 2 * math.pi / 0.001 + 0.01       # RangeNormalize bounds (walk_env.py:364-374, rex_gym_env.py:277-278)
EPISODES, STEPS = 25, 600


def denorm(o):
    o = np.array(o, np.float64)
    o[..., 0:2] *= UA; o[..., 2:4] *= UR; o[..., 4:] *= UA
    return o


def replay_oracle(task, steps=STEPS, episodes=EPISODES, cfg=None, **kw):
    """All episodes side by side (env e replays episode e).  The recorded target_position is a per-episode random draw that
    was not stored; 3.0 (the largest possible) keeps the brake phase out of the window on our side."""
    import ctypes as C
    name = task + "_ol"
    ac, ref = G[name + "_action"][:episodes, :steps], denorm(G[name + "_observ"][:episodes, :steps + 1])
    s = OracleSim(episodes, task, "ol", normalize=True, settle=2, **kw)
    if cfg:
        for k, v in cfg.items():
            setattr(s.cfg, k, v)
        s.L.rexo_destroy(s.h)
        s.h = s.L.rexo_create(C.byref(s.model), C.byref(s.cfg))
    first = denorm(s.reset())
    np.testing.assert_allclose(first, ref[:, 0], atol=2e-5)       # the stored reset observation IS the pristine pose
    out = np.zeros((episodes, steps, ref.shape[2]))
    for t in range(steps):
        o, r, d = s.step(ac[:, t], nthreads=4)
        out[:, t] = denorm(o)
    return out, ref[:, 1:]


def errors(task, **kw):
    ours, ref = replay_oracle(task, **kw)
    rp = np.abs(ours[..., 0:2] - ref[..., 0:2]).max(-1)
    q = np.abs(ours[..., 4:] - ref[..., 4:]).max(-1) if ours.shape[-1] > 4 else np.zeros(rp.shape)
    return rp, q                                                   # [episode][step]


def med(x):
    return float(np.median(x))


def test_gallop_open_loop_tracks_pybullet_over_25_episodes_x_600_steps():
    rp, q = errors("gallop", target_position=3.0)
    # free fall (no contact yet): articulated-body dynamics + motor model alone.  1.5e-5 / 2.6e-5 rad since the link inertias
    # include the compound-shape margin the way Bullet's importer computes them (3.5e-4 / 6e-4 before: tools/compile_urdf.py)
    assert med(q[:, 0]) < 6e-5 and med(q[:, 1]) < 1e-4 and med(rp[:, 1]) < 5e-6
    # touchdown and the first hops
    assert med(q[:, :20].mean(1)) < 1.7e-3 and med(q[:, :20].max(1)) < 3.3e-3 and med(rp[:, :20].max(1)) < 1.4e-3
    # the first 150 control steps (900 sub-steps), the window round 1 pinned
    assert med(q[:, :150].mean(1)) < 3.3e-3 and med(q[:, :150].max(1)) < 2.2e-2
    assert med(rp[:, :150].mean(1)) < 2.4e-3 and med(rp[:, :150].max(1)) < 1.2e-2
    # the error does not grow past step 150: every 150-step window of the 600
    for lo in (150, 300, 450):
        assert med(q[:, lo:lo + 150].mean(1)) < 6.4e-3 and med(q[:, lo:lo + 150].max(1)) < 4.4e-2, lo
        assert med(rp[:, lo:lo + 150].mean(1)) < 5.5e-3 and med(rp[:, lo:lo + 150].max(1)) < 2.5e-2, lo
    # per-episode: at most 1 of the 25 leaves a 0.2 rad tube in 600 steps (measured: none)
    assert np.sum(q.max(1) > 0.2) <= 1


def test_walk_open_loop_tracks_pybullet_over_25_episodes_x_600_steps():
    rp, _ = errors("walk", target_position=3.0, backwards=False)
    assert med(rp[:, :5].max(1)) < 3e-4
    assert med(rp[:, :150].mean(1)) < 1.05e-3 and med(rp[:, :150].max(1)) < 2.8e-3
    assert med(rp.mean(1)) < 2.5e-3 and med(rp.max(1)) < 8.0e-3 and rp.max() < 5.5e-2


def _translation_replay(task, cfg=None, **kw):
    """Replay with our own base position kept: x_ours(t), and F(t) = recorded reward minus OUR non-forward terms ~ x_pybullet / target."""
    import ctypes as C
    ac, R = G[task + "_ol_action"], G[task + "_ol_reward"]
    s = OracleSim(EPISODES, task, "ol", normalize=True, settle=2, target_position=3.0, **kw)
    if cfg:
        for k, v in cfg.items():
            setattr(s.cfg, k, v)
        s.L.rexo_destroy(s.h)
        s.h = s.L.rexo_create(C.byref(s.model), C.byref(s.cfg))
    s.reset()
    X, Rours = np.zeros((EPISODES, STEPS)), np.zeros((EPISODES, STEPS))
    for t in range(STEPS):
        _, r, _ = s.step(ac[:, t], nthreads=4)
        X[:, t] = [-s.env(e).pos[0] for e in range(EPISODES)]
        Rours[:, t] = r
    other = Rours - np.where(X <= 0.05, 0.0, X / 3.0)             # energy + drift + shake terms of our replay (target 3.0, never reached)
    return X, R - other, R


@pytest.mark.parametrize("task,kw", [("gallop", {}), ("walk", dict(backwards=False))])
def test_base_translation_tracks_pybullet_through_the_recorded_rewards(task, kw):
    """The observations carry no base position, but the recorded rewards do (rex_gym_env.py:501-542): the forward term is 0 while
    x <= 0.05 m and x / target afterwards, so (a) the control step at which the reward jumps is the step at which PyBullet's base
    crossed x = 0.05 m -- an absolute event, 47 ... 91 steps into the gallop episodes depending on the stored actions, 116 ... 121
    in walk -- and (b) the size of the jump bounds the episode's (unstored) target, after which every later reward is an absolute
    x.  Measured: our replay crosses within one control step of PyBullet in 24 of 25 gallop episodes (worst 3) and 0-2 steps early
    in walk; x_ours(t) / (x_pybullet(t) / target) is constant over the following ~500 steps to 1.2 % / 2.0 % (std / median,
    median over episodes), and equals the target bounded from the jump within a few percent (median ratio 0.99 / 0.99)."""
    X, F, R = _translation_replay(task, **kw)
    t_rec = np.array([int(np.argmax(R[e] > 0.01)) for e in range(EPISODES)])
    t_our = np.array([int(np.argmax(X[e] > 0.05)) for e in range(EPISODES)])
    assert np.all(R[np.arange(EPISODES), t_rec - 1] < 0.002) and np.all(R[np.arange(EPISODES), t_rec] > 0.012)     # a jump, not a ramp
    d = t_our - t_rec
    assert np.abs(d).max() <= 3 and np.sum(np.abs(d) <= 1) >= (22 if task == "gallop" else 18) and abs(np.median(d)) <= 1, d
    if task == "gallop":
        assert t_rec.max() - t_rec.min() > 30                      # the event time is episode-specific, and reproduced episode by episode
        assert np.corrcoef(t_rec, t_our)[0, 1] > 0.99
    cv, ratio = [], []
    for e in range(EPISODES):
        m = (np.arange(STEPS) > t_rec[e] + 10) & (F[e] > 0.02) & (F[e] < 0.9)
        implied = X[e, m] / F[e, m]                                # = target if x_ours == x_pybullet
        cv.append(implied.std() / np.median(implied))
        lo = 0.05 / F[e, t_rec[e]]                                 # x in (0.05, 0.05 + one step's travel] at the jump
        hi = lo * (1 + (X[e, t_rec[e]] - X[e, t_rec[e] - 1]) / 0.05)
        ratio.append(np.median(implied) / (0.5 * (lo + hi)))
    cv, ratio = np.array(cv), np.array(ratio)
    assert np.median(cv) < 0.03 and cv.max() < 0.07, (np.median(cv), cv.max())
    assert 0.97 < np.median(ratio) < 1.03 and ratio.min() > 0.85 and ratio.max() < 1.12, ratio


def test_walk_open_loop_to_the_goal_brake_and_standstill_like_pybullet():
    """Four recorded walk-ol episodes over 1200 control steps = 6 s: ramp up, walk 1.0-1.8 m to the goal, brake, stand still.
    The goal is a per-episode random draw that was not stored; it is recovered from the recording itself -- the forward reward
    jumps from 0 to x / target when x passes 0.05 m (rex_gym_env.py:516-520), so target = 0.05 m (+ at most one step's travel)
    / jump.  With that target the open-loop replay reproduces what no observation channel carries: the step at which PyBullet's
    base passed target + 0.15 m (the reward drops from 1 to target - x, :512-513) within 15 control steps after 450-620, and the
    place where the robot finally stands, target + 0.29 ... 0.37 m recorded, within 2 cm; roll / pitch stay within a few mrad of
    the recording through all three phases."""
    ac, ob, rw = G["walk_ol_long_action"], denorm(G["walk_ol_long_observ"]), G["walk_ol_long_reward"]
    for k in range(ac.shape[0]):
        # the target from the jump: replay the first 200 steps once to know our own step travel at the crossing (~1 mm)
        probe = OracleSim(1, "walk", "ol", normalize=True, settle=2, target_position=3.0, backwards=False)
        probe.reset()
        xs = []
        for t in range(200):
            probe.step(ac[k:k + 1, t]); xs.append(-probe.env(0).pos[0])
        t_jump = int(np.argmax(rw[k] > 0.01))
        assert rw[k, t_jump - 1] < 0.002 < 0.012 < rw[k, t_jump] and abs(int(np.argmax(np.array(xs) > 0.05)) - t_jump) <= 2
        lo = 0.05 / (rw[k, t_jump] - rw[k, t_jump - 1])           # the other reward terms do not jump
        target = lo * (1 + 0.5 * (xs[t_jump] - xs[t_jump - 1]) / 0.05)
        assert 0.95 < target < 1.9
        s = OracleSim(1, "walk", "ol", normalize=True, settle=2, target_position=float(target), backwards=False)
        s.reset()
        R, P = [], []
        for t in range(1200):
            o, r, d = s.step(ac[k:k + 1, t])
            assert not d[0], (k, t)
            R.append(float(r[0])); P.append(denorm(o)[0, :2])
        R, P = np.array(R), np.array(P)
        drop_rec, drop_our = int(np.argmax(np.diff(rw[k]) < -0.5)), int(np.argmax(np.diff(R) < -0.5))
        assert 400 < drop_rec < 650 and abs(drop_our - drop_rec) <= 15, (k, drop_rec, drop_our)      # measured: ours 5, 8, 6, 6 steps early
        assert rw[k, -1] < -0.25 and abs(R[-1] - rw[k, -1]) < 0.02, (k, R[-1], rw[k, -1])             # stands where PyBullet's stands (measured: within 1.3 cm after 1.4-2.1 m)
        assert abs(R[-1] - R[-100]) < 2e-3 and abs(rw[k, -1] - rw[k, -100]) < 2e-3                   # ... and both stand still
        err = np.abs(P - ob[k, 1:, :2]).max(1)
        assert err[:400].mean() < 3e-3 and err[400:800].mean() < 8e-3 and err[800:].mean() < 9e-3, (k, err[:400].mean(), err[400:800].mean(), err[800:].mean())
        assert np.abs(R[drop_rec + 60:] - rw[k, drop_rec + 60:]).mean() < 0.03


def test_turn_open_loop_recordings_in_yaw_invariant_quantities():
    """The 25 recorded turn-ol episodes (160 steps) were called unusable in round 1 ("disagree from step 1").  Read against
    turn_env.py:129-160,271-311 the reason is mostly bookkeeping: every episode starts at a yaw drawn from U(0.2, 6) that the
    observation does not carry, the observation's two rate channels are WORLD-frame components (rex.py:548-558) and so rotate
    with that yaw, and the left / right pose table is selected by (init, target) yaw, also not stored.  Compared in what does
    not depend on the yaw -- roll, pitch (Euler angles of R = Rz Ry Rx) and the horizontal rate magnitude -- and with the
    turning direction chosen per episode by the better fit over the first 40 steps (12-13 of 25 come out clockwise, as a fair
    draw would), the replay tracks the recordings: roll / pitch 7e-4 rad after the first step, 5e-3 over the first 40 steps,
    1.4e-2 over all 160 -- three to eight times looser than walk-ol, with a 25 % mismatch of the first step's pitch rate
    (0.22 rad/s recorded) that the unknown June-2020 pose table could explain but nothing here can confirm."""
    ac, ob = G["turn_ol_action"], denorm(G["turn_ol_observ"])
    ref_rp, ref_w = ob[:, 1:, 0:2], np.hypot(ob[:, 1:, 2], ob[:, 1:, 3])
    err = {}
    for to, io in ((1.0, 3.0), (3.0, 1.0)):                       # clockwise / counter-clockwise (turn_env.py:313-322)
        s = OracleSim(EPISODES, "turn", "ol", normalize=True, settle=2, target_orient=to, init_orient=io)
        s.reset()
        cw = s.env(0).clockwise
        out = np.array([denorm(s.step(ac[:, t], nthreads=4)[0]) for t in range(160)]).transpose(1, 0, 2)
        err[cw] = (np.abs(out[..., 0:2] - ref_rp).max(-1), np.abs(np.hypot(out[..., 2], out[..., 3]) - ref_w))
    pick = err[1][0][:, :40].mean(1) < err[0][0][:, :40].mean(1)
    rp = np.where(pick[:, None], err[1][0], err[0][0])
    w = np.where(pick[:, None], err[1][1], err[0][1])
    assert 6 <= pick.sum() <= 19                                   # both directions occur
    assert med(rp[:, 0]) < 1.2e-3 and med(rp[:, :40].mean(1)) < 8e-3 and med(rp.mean(1)) < 2.2e-2
    assert med(w[:, 0]) < 0.09 and med(ref_w[:, 0]) > 0.15          # first-step pitch rate: 0.22 recorded, ours within 0.054


def _standup_replay(steps, episodes=EPISODES):
    ac, ref, rw = G["standup_ol_action"][:episodes], denorm(G["standup_ol_observ"][:episodes]), G["standup_ol_reward"][:episodes]
    s = OracleSim(episodes, "standup", "ol", normalize=True)      # the full reset hold (rex.py:314-323), not the pristine pose
    s.reset()
    st = s.state(0)
    P, R = [], []
    for t in range(steps):
        o, r, _ = s.step(ac[:, t], nthreads=4)
        P.append(denorm(o)[:, 1]); R.append(r.copy())
    return np.array(P).T, np.array(R).T, ref[:, 1:steps + 1, 1], rw[:, :steps], st, ref[:, 0]


def test_standup_reset_hold_ends_like_the_recorded_one():
    """Standup episodes start from whatever the 600-sub-step reset hold (rex.py:314-323: 100 x `stand`, 500 x `rest_position`
    with the foot command at 6 rad, far beyond the 2.59 rad limit) leaves behind.  What the recordings and the README animation
    (images/standup_ol.gif, first frame) say about that state: the robot rests ON ITS FOLDED FEET with the trunk clear of the
    ground, and it is STILL MOVING when the episode starts (recorded reset observation: pitch -0.0097 rad, pitch rate
    -0.047 rad/s in all 25 episodes); the first reward -0.184 = -(|x| + |y| + 0.21 - z) after one control step.  With the two
    Bullet behaviours restated this round (the saturated foot motors whip the 1.9e-4 kg m^2 feet at > 100 rad/s, the clamp caps
    that, the joint overshoots the limit by > 0.04 rad and the split-impulse branch then never pushes it back) the hold ends
    at z = 0.054, feet at 2.69-2.72 rad, pitch -0.007, pitch rate -0.058 -- creeping like the recorded one; round 1's model
    sat still on its toes at z = 0.0657 with the feet exactly on the limit (first reward -0.160)."""
    P, R, pref, rref, st, ob0 = _standup_replay(1)
    assert 2.62 < st["q"][2] < 2.80 and 2.62 < st["q"][8] < 2.80                 # past the 2.59 rad limit, front and rear
    pitch = 2 * st["quat"][1]
    assert abs(pitch - med(ob0[:, 1])) < 6e-3                                   # recorded -0.0097
    assert -0.09 < st["angvel"][1] < -0.02 and -0.06 < med(ob0[:, 3]) < -0.03    # still creeping, same sign and size
    assert np.abs(R[:, 0] - rref[:, 0]).max() < 0.016                            # first reward: ours -0.197, recorded -0.184


def test_standup_hop_tracks_pybullet_through_the_first_30_steps():
    """From our own hold the hop off the folded legs (first 30 control steps = 150 sub-steps, saturated motors, open loop)
    keeps the recorded pitch within 0.07 rad (the trace has the recorded shape, about one control step early) and crosses
    |pos - target| = 0.1 (reward sign flip) within two control steps of PyBullet; the rate at which the reward rises over the
    first 10 steps (the trunk being lifted) matches the recorded one within 15 %."""
    P, R, pref, rref, _, _ = _standup_replay(30)
    err = np.abs(P - pref).max(1)
    assert med(err) < 0.07 and err.max() < 0.085
    flip = np.abs(np.argmax(R > 0, axis=1) - np.argmax(rref > 0, axis=1))
    assert flip.max() <= 2
    rise, rise_ref = R[:, 9] - R[:, 0], rref[:, 9] - rref[:, 0]
    assert np.abs(rise / rise_ref - 1).max() < 0.15


@pytest.mark.xfail(reason="DESIGN.md sections 3 and 9: after the hop our robot pitches nose-down in flight (-3.4 rad/s against the "
                          "recorded -0.5 rad/s) and falls at step ~95; PyBullet's lands and stands for the remaining 360 steps at reward "
                          "0.98.  The outcome flips between foot joints at 2.68 and 2.69 rad when the episode starts (next test); our "
                          "hold ends at 2.71 / 2.69 because the limit rows creep while the solver sits at its iteration cap.", strict=False)
def test_standup_episode_stands_like_the_recorded_ones():
    P, R, pref, rref, _, _ = _standup_replay(200)
    assert med(R[:, 199]) > 0.9 and med(rref[:, 199]) > 0.9


def test_standup_outcome_is_decided_by_the_foot_angle_the_hold_ends_in():
    """The sensitivity behind the xfail above, pinned: the same replay started with the four foot joints at 2.66 rad (0.03-0.05
    rad less folded than our hold leaves them, everything else untouched) hops, lands and stands like the 25 recorded episodes --
    reward 0.97 at step 119 (recorded 0.97), pitch within 0.1 rad of the recorded one at steps 60 and 100 -- and at 2.70 rad it falls.
    The hold reaches 2.68 / 2.66 when the feet stop at the velocity clamp and creeps on from there while the solver runs at its
    60-iteration cap (PyBullet's recorded reset observation is creeping too): with 300 iterations it stays at 2.680 / 2.661."""
    ac, ref, rw = G["standup_ol_action"][:6], denorm(G["standup_ol_observ"][:6]), G["standup_ol_reward"][:6]
    out = {}
    for feet in (2.66, 2.70):
        s = OracleSim(6, "standup", "ol", normalize=True)
        s.reset()
        for i in range(6):
            e = s.env(i)
            for leg in range(4):
                e.q[3 * leg + 2] = feet; e.qd[3 * leg + 2] = 0.0
        P, R = [], []
        for t in range(120):
            o, r, _ = s.step(ac[:, t], nthreads=4)
            P.append(denorm(o)[:, 1]); R.append(r.copy())
        out[feet] = (np.array(P).T, np.array(R).T)
    P, R = out[2.66]
    assert med(R[:, 119]) > 0.9 and abs(med(R[:, 119]) - med(rw[:, 119])) < 0.05
    assert abs(med(P[:, 59]) - med(ref[:, 60, 1])) < 0.1 and abs(med(P[:, 99]) - med(ref[:, 100, 1])) < 0.1
    assert med(out[2.70][1][:, 119]) < 0.0
    s = OracleSim(1, "standup", "ol", normalize=True, solver_iterations=300)
    s.reset()
    q = s.state(0)["q"]
    assert abs(q[2] - 2.680) < 4e-3 and abs(q[8] - 2.661) < 4e-3


def _mean_joint_error(steps=100, episodes=12, **ov):
    ours, ref = replay_oracle("gallop", steps=steps, episodes=episodes, cfg=ov, target_position=3.0)
    return float(np.median(np.abs(ours[..., 4:] - ref[..., 4:]).max(-1).mean(1)))


def test_recorded_trajectories_identify_the_friction_coefficient():
    """URDF link default 0.5 x plane.urdf lateral_friction 1.0 = 0.5; `<contact_coefficients mu="100">` (rex.urdf:194) is
    ignored by Bullet's URDF parser.  The recorded hopping is sharply selective: any other value is several times worse."""
    base = _mean_joint_error()
    for mu in (0.25, 1.0):
        other = _mean_joint_error(friction=mu)
        assert other > 2.5 * base, (mu, other, base)
    for mu in (0.45, 0.55):
        assert _mean_joint_error(steps=300, episodes=25, friction=mu) > 1.15 * _mean_joint_error(steps=300, episodes=25), mu
    # the base translation read off the recorded rewards is sharper still: mean distance (control steps) between our and
    # PyBullet's x = 0.05 m crossing over the 25 gallop episodes -- 0.52 at 0.5; 2.4 / 1.7 at 0.45 / 0.55; 7.3 / 6.4 at 0.35 / 1.0

    def crossing_error(mu):
        X, _, R = _translation_replay("gallop", cfg=dict(friction=mu))
        t_rec = np.array([int(np.argmax(R[e] > 0.01)) for e in range(EPISODES)])
        t_our = np.array([int(np.argmax(X[e] > 0.05)) for e in range(EPISODES)])
        return float(np.abs(t_our - t_rec).mean())
    e_half = crossing_error(0.5)
    assert e_half < 0.9 and crossing_error(0.45) > 2.5 * e_half and crossing_error(0.55) > 2.0 * e_half


def test_recorded_trajectories_select_the_link_damping_and_the_toe_reach():
    """Bullet's damping on every link (0.04) and the effective toe reach (-0.25 mm) are the values the 25 recorded episodes
    prefer over their neighbours.  Damping: mean roll/pitch error over all episodes x 300 steps, 5.0e-3 rad at 0.04 against
    5.7e-3 without and 6.1e-3 at 0.2 (the base angular velocity error moves the same way).  Toe reach: mean joint error of the
    20 touchdown steps, 1.9e-3 rad at -0.25 mm against 3.0e-3 for the exact hull and 7.2e-3 with Bullet's 1 mm importer margin."""
    import oracle.oracle as O

    def pitch_err(**ov):
        ours, ref = replay_oracle("gallop", steps=300, cfg=ov, target_position=3.0)
        return float(np.abs(ours[..., 0:2] - ref[..., 0:2]).max(-1).mean())
    base = pitch_err()
    assert pitch_err(link_damping=0.0) > 1.08 * base and pitch_err(link_damping=0.2) > 1.15 * base
    saved = O.TOE_MARGIN
    try:
        e_0 = _mean_joint_error(steps=20, episodes=25)

        def crossing_error():                        # independent observable: the x = 0.05 m crossing read off the rewards
            X, _, R = _translation_replay("gallop")
            return float(np.abs(np.array([int(np.argmax(X[e] > 0.05)) - int(np.argmax(R[e] > 0.01)) for e in range(EPISODES)])).mean())
        c_0 = crossing_error()                       # 0.52 control steps; 0.88 for the exact hull, 1.92 with the importer margin
        for m in (0.0, 0.001):                       # the exact hull / Bullet's 1 mm importer margin
            O.TOE_MARGIN = m
            e_m = _mean_joint_error(steps=20, episodes=25)
            assert e_m > 1.3 * e_0, (m, e_m, e_0)
            assert crossing_error() > (1.3 if m == 0.0 else 2.5) * c_0, m
    finally:
        O.TOE_MARGIN = saved


def test_fixture_matches_the_reference_checkpoints():
    """The fixture is the checkpoints' EpisodeMemory: compared with the rows of the same memory variables that
    tests/golden/tf_memory_golden.npz samples from the first 400 steps of the same checkpoints (tools/gen_policy_golden.py)."""
    M = np.load(os.path.join(os.path.dirname(__file__), "golden", "tf_memory_golden.npz"))
    for task in ("gallop", "walk", "turn", "standup"):
        name = task + "_ol"
        n = G[name + "_action"].shape[1]
        ep, t = np.divmod(M[name + "_rows"], 400)
        assert G[name + "_observ"].shape[0] == 25 and ep.max() == 24
        k = t <= n
        np.testing.assert_array_equal(G[name + "_observ"][ep[k], t[k]], M[name + "_observ"][k])
        k = t < n
        assert k.sum() >= 400, (task, k.sum())
        np.testing.assert_array_equal(G[name + "_action"][ep[k], t[k]], M[name + "_action"][k])
        np.testing.assert_array_equal(G[name + "_reward"][ep[k], t[k]], M[name + "_reward"][k])


def _ripple_period(x, lo=5):
    x = x - x.mean()
    spec = np.abs(np.fft.rfft(x * np.hanning(len(x))))
    return len(x) / (int(np.argmax(spec[lo:])) + lo)


def test_wall_clock_gait_of_the_recorded_walk_ik_episodes():
    """GaitPlanner.loop reads time.time() (gait_planner.py:108-110).  The walk-ik episodes stored in the shipped checkpoint
    show what that meant in training: the trunk PITCH ripples with a period of 8.0 control steps and the ROLL with 15.4-16.7 --
    a trot rocks sideways once and nods twice per gait cycle, so the cycle lasted ~16 control steps = 80 ms of simulation time
    instead of the nominal 0.65 s: the wall clock ran ~9x faster than the simulation (a 16-step cycle needs a scale in
    [8.6, 9.2); 45 ms of wall time per batched control step, the same machine speed the gallop-ik recording implies below).
    [Round 1 and most of round 2 read the 8-step pitch ripple as the gait cycle and concluded x16; the base translation
    recovered from the recorded rewards settled it: at x16 the restated robot needs 236-282 steps to cover its first 5 cm,
    PyBullet's needed 143-186.]  At gait_clock_scale = 9 the restatement reproduces the recorded regime: pitch ripple period
    8.0 (recorded 8.0), pitch ripple size within 25 % (3.5e-3 vs 4.1e-3 rad), roll ripple half the recorded size, level walk
    (|roll|, |pitch| < 0.04 for the whole window), and the x = 0.05 m crossing -- read off the recorded rewards like in
    test_base_translation_tracks_pybullet_through_the_recorded_rewards -- inside the recorded range (ours 158-167, recorded
    143-186).  With the simulation clock (scale 1) the same actions give the nominal trot, which is a different motion
    altogether (and tips over in this model, DESIGN.md section 2)."""
    ref, ac, rw = denorm(G["walk_ik_observ"]), G["walk_ik_action"], G["walk_ik_reward"]
    np.testing.assert_array_equal(ref[:, 0], 0.0)                       # pristine reset observation
    n = ref.shape[0]
    p_rec = [_ripple_period(ref[e, 100:300, 1]) for e in range(n)]
    r_rec = [_ripple_period(ref[e, 100:300, 0]) for e in range(n)]
    assert all(7.5 < p < 8.5 for p in p_rec) and all(14.5 < r < 17.5 for r in r_rec), (p_rec, r_rec)     # nods twice per cycle
    cross_rec = np.array([int(np.argmax(rw[e] > 0.01)) for e in range(n)])
    assert 130 < cross_rec.min() and cross_rec.max() < 200

    def replay(scale, steps=300):
        s = OracleSim(n, "walk", "ik", normalize=True, settle=2, target_position=3.0, backwards=False, gait_clock_scale=scale)
        s.reset()
        out, cross = [], np.full(n, -1)
        for t in range(steps):
            o, r, d = s.step(ac[:, t], nthreads=4)
            assert not d.any(), (scale, t)
            out.append(denorm(o))
            for e in range(n):
                if cross[e] < 0 and -s.env(e).pos[0] > 0.05:
                    cross[e] = t
        return np.array(out).transpose(1, 0, 2), cross
    out, cross = replay(9.0)
    for e in range(n):
        assert abs(_ripple_period(out[e, 100:, 1]) - p_rec[e]) < 0.5                 # pitch ripple: same period ...
        assert 0.7 < out[e, 100:, 1].std() / ref[e, 101:301, 1].std() < 1.3           # ... and size (measured 0.78-0.92)
        assert 0.25 < out[e, 100:, 0].std() / ref[e, 101:301, 0].std() < 1.5          # roll ripple: 0.3-0.55 of the recorded one
    assert np.abs(out[:, :, :2]).max() < 0.04                                        # level for the whole window (recorded: < 0.02)
    assert cross_rec.min() - 5 <= cross.min() and cross.max() <= cross_rec.max() + 5, (cross, cross_rec)
    _, cross16 = replay(16.0)
    assert cross16.min() > cross_rec.max() + 30                                      # x16 shuffles on the spot: too slow by half
    s = OracleSim(1, "walk", "ik", normalize=True, settle=2, target_position=2.0, backwards=False)      # simulation clock
    s.reset()
    big = 0.0
    for t in range(200):
        o, r, d = s.step(ac[0, t][None, :])
        big = max(big, float(np.abs(denorm(o[0])[:2]).max()))
        if d[0]:
            break
    assert big > 0.1                                                     # the nominal trot rocks the base 25x more


def test_wall_clock_gait_of_the_recorded_gallop_ik_episodes():
    """Same wall-clock effect on the gallop-ik policy's training data, where the observation also carries the 12 joint angles:
    the recorded leg-joint ripple has a 7.0 control-step period (0.3 s gait period / 42 ms => the wall clock ran ~7.1x
    faster than the simulation).  At gait_clock_scale = 8.5 (7-step cycle) the restatement reproduces period and size of the
    joint-angle ripple (leg 0.059 rad, foot 0.046 rad recorded) -- IK-driven legs through the motor model at 24 Hz.
    What this regime does NOT determine is where the robot goes: the recorded forward reward is 0 on every one of the 1000
    steps of every episode (PyBullet's base never got past x = 0.05 m -- the shipped gallop-ik policy was trained on a robot
    hopping on the spot or backwards), and in the restatement the net drift of the 24 Hz shuffle is an aliasing effect
    between gait clock and control step: +0.58 m in 600 steps at scale 8.25, -0.63 m at 9.5, with the real clock jittering
    in between.  A constant scale cannot reproduce that, and the test only records the fact."""
    ref = denorm(G["gallop_ik_observ"])
    ac = G["gallop_ik_action"]
    assert G["gallop_ik_reward"].max() <= 0.0                       # forward term never positive: x <= 0.05 m throughout
    drift = {}
    for sc in (8.25, 9.5):
        s = OracleSim(3, "gallop", "ik", normalize=True, settle=2, target_position=3.0, gait_clock_scale=sc)
        s.reset()
        for t in range(600):
            s.step(ac[:, t], nthreads=3)
        drift[sc] = np.array([-s.env(e).pos[0] for e in range(3)])
    assert drift[8.25].min() > 0.3 and drift[9.5].max() < -0.3, drift     # same 7-step ripple, opposite directions
    scale = 8.5      # phase step 6 ms * 8.5 / 0.3 s = 0.17 per control step: phi >= 0.99 after 6 steps, +1 step for the restart = 7
    for ep in range(3):
        s = OracleSim(1, "gallop", "ik", normalize=True, settle=2, target_position=2.0, gait_clock_scale=scale)
        s.reset()
        out = []
        for t in range(400):
            o, r, d = s.step(ac[ep, t][None, :])
            assert not d[0], (ep, t)
            out.append(denorm(o[0]))
        out = np.array(out)

        def period(x):
            x = x - x.mean()
            spec = np.abs(np.fft.rfft(x)); k = int(np.argmax(spec[5:])) + 5
            return len(x) / k
        assert abs(period(ref[ep, 101:401, 5]) - 7.0) < 0.5 and abs(period(out[100:, 5]) - 7.0) < 1.0
        for j in (5, 6, 11, 12):                                       # leg / foot joints of a front and a rear leg
            ours, real = out[100:, j].std(), ref[ep, 101:401, j].std()
            assert 0.6 * real < ours < 1.6 * real, (ep, j, ours, real)
        assert abs(out[100:, 1].mean() - ref[ep, 101:401, 1].mean()) < 0.03      # mean pitch of the hopping gait


def test_shipped_gallop_policy_closes_the_loop_like_its_training_runs():
    """End to end: the gallop-ol policy the reference ships (TF checkpoint -> pure-Python reader -> numpy restatement of
    ForwardGaussianPolicy + StreamingNormalize) drives the restated simulator.  It gallops forward (-x) for the whole
    1000-step episode, and its progress is consistent with the rewards PyBullet produced during training: the forward
    reward is x / target with target ~ U(1, 3) (gallop_env.py:151, rex_gym_env.py:513-520), so every recorded reward implies
    a target x_ours(t) / reward(t), which has to fall in that range if the two simulators cover ground at the same rate."""
    from oracle import agent_oracle as AO
    from rex_gym_b200.agents.networks import read_tf_policy
    w, filt = read_tf_policy(os.path.join(os.path.dirname(__file__), "golden", "policies", "gallop", "ol"))
    f = AO.StreamingNormalize((16,), True, True, 5)
    f.count, f.mean, f.var_sum = filt[0], np.array(filt[1], np.float64), np.array(filt[2], np.float64)
    s = OracleSim(1, "gallop", "ol", normalize=True, settle=2, target_position=2.0)
    obs = s.reset()
    e = s.env(0)
    xs = []
    for t in range(1000):
        _, mean, _, _ = AO.perform(w, f, obs.astype(np.float64), False)
        obs, r, d = s.step(mean.astype(np.float32))
        xs.append(e.pos[0])
        assert not d[0], t
    xs = -np.array(xs)
    assert 0.75 < xs[499] < 1.3 and 1.6 < xs[999] < 2.6 and abs(e.pos[1]) < 0.3          # ~0.35 m/s, straight
    implied = xs[149] / G["gallop_ol_reward"][:, 149]                                       # recorded: sampled actions, 25 episodes
    assert np.sum((implied > 0.85) & (implied < 3.5)) >= 21, implied


def test_shipped_walk_policy_reproduces_the_recorded_reward_profile():
    """The shipped walk-ol policy in closed loop on the restated simulator, target 2.0 m: ramps up, walks to the goal, brakes
    and stands still -- the per-step reward (rex_gym_env.py:501-542) has the profile of the 25 episodes PyBullet recorded in
    the checkpoint: r(400)/r(200) in [3.8, 4.6] (acceleration phase), a final plateau of -0.28 ... -0.41 (the robot needs
    0.3-0.4 m to stop past the goal: `tp - cx` once cx > tp + 0.15), and standing still for the rest of the 2000 steps."""
    from oracle import agent_oracle as AO
    from rex_gym_b200.agents.networks import read_tf_policy
    w, filt = read_tf_policy(os.path.join(os.path.dirname(__file__), "golden", "policies", "walk", "ol"))
    f = AO.StreamingNormalize((4,), True, True, 5)
    f.count, f.mean, f.var_sum = filt[0], np.array(filt[1], np.float64), np.array(filt[2], np.float64)
    s = OracleSim(1, "walk", "ol", normalize=True, settle=2, target_position=2.0, backwards=False)
    obs = s.reset()
    e = s.env(0)
    R, X = [], []
    for t in range(2000):
        _, mean, _, _ = AO.perform(w, f, obs.astype(np.float64), False)
        obs, r, d = s.step(mean.astype(np.float32))
        R.append(float(r[0])); X.append(e.pos[0])
        assert not d[0], t
    R, X = np.array(R), -np.array(X)
    assert 3.6 < R[400] / R[200] < 4.8                       # recorded: 3.76 ... 4.57
    assert 0.9 < X[400] < 1.2                                # recorded r(400) = x / target, e.g. 0.96 at target ~1.1
    assert -0.45 < R[-1] < -0.25 and abs(R[-1] - R[1200]) < 0.03      # recorded plateau: -0.414 ... -0.278, reached by step ~800
    assert abs(X[-1] - X[1200]) < 0.02 and 2.2 < X[-1] < 2.5          # stands still past the goal
