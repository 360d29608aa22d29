"""TD3 (twin critics, target policy smoothing, delayed policy updates; no reference code, DESIGN.md section 6.14).

Without a GPU: argument rejection by the three ss_td3_targets* entry points, the constructors' and the checkpoint loader's
ValueErrors, the cross-rank agreement on the TD3 options under gloo, and the header constants against _lib.py.
On the GPU, compared with ==: the new targets against ss_ddpg_targets* with one critic and no smoothing, default-valued
options against no options, the rollout, the delayed updates and checkpoint resume.  Against the torch autograd
restatement (tests/td3_oracle.py on oracle/learner_oracle.py): the float32 target with the host Philox draws
(tests/philox_ref.py), the tensor-core targets against the float32 ones, six TD3 updates, and the statistics of the smoothing noise."""
import json
import os
import re
import socket
import time

import numpy as np
import pytest
import torch

from oracle import learner_oracle as lo
from tests import philox_ref
from tests import td3_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 1 << 20              # a 16-byte aligned stand-in for a device pointer: every call below is refused before any use


def _lib():
    from skillshot_learning_b200 import _lib
    return _lib


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def _td3_calls(L):
    """(name, call(**overrides)) for each entry point; every default argument is valid"""
    def f32(ta=P, tc=P, tc2=P, frames=4, r=P, s2=P, gamma=0.99, sd=0.2, clip=0.5, row_offset=0, y=P, n=16):
        return L.ss_td3_targets_frames(ta, tc, tc2, frames, r, s2, None, gamma, sd, clip, 1, 2, row_offset, y, n, None, 0, None)

    def tc(ta=P, tc=P, tc2=P, frames=1, r=P, s2=P, gamma=0.99, sd=0.2, clip=0.5, row_offset=0, y=P, n=16):
        assert frames == 1
        return L.ss_td3_targets_tc(ta, tc, tc2, r, s2, None, gamma, sd, clip, 1, 2, row_offset, y, n, P, 1 << 20, None)

    def ftc(ta=P, tc=P, tc2=P, frames=4, r=P, s2=P, gamma=0.99, sd=0.2, clip=0.5, row_offset=0, y=P, n=16):
        return L.ss_td3_targets_frames_tc(ta, tc, tc2, frames, r, s2, None, gamma, sd, clip, 1, 2, row_offset, y, n, P, 1 << 30,
                                          None)
    return [("frames", f32), ("tc", tc), ("frames_tc", ftc)]


@pytest.mark.parametrize("which", ["frames", "tc", "frames_tc"])
def test_td3_target_entry_points_reject_bad_arguments(which):
    L = _lib().lib
    call = dict(_td3_calls(L))[which]
    for k in ("ta", "tc", "r", "s2", "y"):
        assert call(**{k: None}) == -1, k
    for n in (0, -5):
        assert call(n=n) == -1
    assert call(sd=-0.1) == -1 and call(sd=float("nan")) == -1
    assert call(clip=-0.5) == -1
    assert call(row_offset=-1) == -1
    if which != "tc":
        for f in ((0, 21, -1) if which == "frames" else (0, 1, 21)):
            assert call(frames=f) == -1, f
    if which != "frames":
        assert call(ta=P + 8) == -1 and call(tc2=P + 4) == -1          # misaligned parameter vectors
    if which == "tc":
        assert L.ss_td3_targets_tc(P, P, P, P, P, None, 0.9, 0.2, 0.5, 1, 2, 0, P, 16, P, 64, None) == -1     # short workspace
        assert L.ss_td3_targets_tc(P, P, P, P, P, None, 0.9, 0.2, 0.5, 1, 2, 0, P, 16, None, 1 << 20, None) == -1
    if which == "frames_tc":
        assert L.ss_td3_targets_frames_tc(P, P, None, 4, P, P, None, 0.9, 0.2, 0.5, 1, 2, 0, P, 16, P, 1024, None) == -1


def test_header_constants_match_the_python_mirror():
    _l = _lib()
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    assert int(re.search(r"#define\s+SS_TAG_TARGET_NOISE\s+(\d+)", text).group(1)) == _l.TAG_TARGET_NOISE
    rng_h = open(os.path.join(ROOT, "skillshot_learning_b200", "csrc", "ss_rng.cuh")).read()
    assert int(re.search(r"kTagTargetNoise\s*=\s*(\d+)", rng_h).group(1)) == _l.TAG_TARGET_NOISE
    tags = [int(t) for t in re.findall(r"constexpr uint32_t kTag\w+\s*=\s*(\d+)", rng_h)]
    assert len(tags) == len(set(tags))                                  # a tag of its own
    body = re.search(r"#define\s+SS_TD3_TC_WORKSPACE_BYTES\(n\)\s+(.*)", text).group(1)
    expr = body.replace("(int64_t)", "").replace("/", "//")
    for n in (1, 3, 4, 1000, 65536, 65537):
        assert eval(expr, {"n": n}) == _l.td3_tc_workspace_bytes(n), n


@pytest.mark.parametrize("kw", [dict(policy_delay=0), dict(policy_delay=-2), dict(policy_delay=1.5), dict(target_noise=-0.1),
                                dict(target_noise_clip=-1e-3), dict(target_noise=float("nan"))])
def test_constructors_reject_bad_td3_options_before_allocating(kw):
    from skillshot_learning_b200 import ActorCritic, SelfPlayTrainer
    with pytest.raises(ValueError):
        ActorCritic(device="cuda:0", **kw)
    with pytest.raises(ValueError):
        SelfPlayTrainer(64, device="cuda:0", **kw)


def _bare_learner(twin):
    """An ActorCritic with only what check_state_dict reads (no device needed)"""
    from skillshot_learning_b200 import ActorCritic
    from skillshot_learning_b200.learner import A_N, C_N
    ac = ActorCritic.__new__(ActorCritic)
    ac.twin_critics = twin
    c_off = (A_N + 3) // 4 * 4
    total = c_off + C_N if not twin else (c_off + C_N + 3) // 4 * 4 + C_N
    ac.params = torch.zeros(total)
    return ac


def test_checkpoint_refusals_on_a_hand_built_state_dict():
    single, twin = _bare_learner(False), _bare_learner(True)
    sd1 = dict(params=torch.zeros(single.params.numel()), step_actor=0, step_critic=0, counter=0, seed=0)
    sd2 = dict(params=torch.zeros(twin.params.numel()), step_actor=0, step_critic=0, step_critic2=0, td3_updates=3, counter=0, seed=0)
    with pytest.raises(ValueError, match="one critic does not load into a learner with twin critics"):
        twin.check_state_dict(sd1)
    with pytest.raises(ValueError, match="twin critics does not load into a learner with one critic"):
        single.check_state_dict(sd2)
    single.check_state_dict(sd1)
    twin.check_state_dict(sd2)


# ---- the agreement of the ranks on the TD3 options (gloo, world size 2, under a timeout) -----------------------------
WORLD = 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_case(rank, case):
    import torch.distributed as dist
    from skillshot_learning_b200 import ActorCritic
    from skillshot_learning_b200.learner import check_td3_options
    try:
        if case == "delay":          # the learner's constructor: rank 1 passes another policy_delay
            ActorCritic(device="cpu", process_group=True, twin_critics=True, policy_delay=1 + rank)
        elif case == "refuse":
            check_td3_options(True, 2, -0.2 if rank == 1 else 0.2, 0.5, True)
        else:
            check_td3_options(True, 2, 0.2, 0.5, True)
    except (ValueError, RuntimeError) as e:
        msg = "%s: %s" % (type(e).__name__, e)
    else:
        msg = None
    dist.barrier()
    return msg


def _worker(rank, case, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(WORLD))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        out = _gloo_case(rank, case)
        with open(os.path.join(out_dir, "%s_%d.json" % (case, rank)), "w") as f:
            json.dump(out, f)
    finally:
        dist.destroy_process_group()


def _run(case, tmp_path, timeout=120.0):
    import torch.multiprocessing as mp
    ctx = mp.spawn(_worker, args=(case, _free_port(), str(tmp_path)), nprocs=WORLD, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=1.0):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("a rank did not finish within %.0f s" % timeout)
    return [json.load(open(tmp_path / ("%s_%d.json" % (case, r)))) for r in range(WORLD)]


def test_ranks_refuse_a_mismatched_policy_delay_together(tmp_path):
    m0, m1 = _run("delay", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 passed policy_delay = 2, rank 0 1"


def test_ranks_raise_together_when_one_refuses_its_options(tmp_path):
    m0, m1 = _run("refuse", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 refused: target_noise must be >= 0, got -0.2"


def test_equal_td3_options_agree(tmp_path):
    assert _run("agree", tmp_path) == [None, None]


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _nets(frames, seed=0):
    rng = np.random.default_rng(seed)
    theta, phi, phi2 = lo.init_actor(rng, frames), lo.init_critic(rng, frames), lo.init_critic(rng, frames)
    dev = torch.device("cuda:0")
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    return rng, theta, phi, phi2, t


def _batch(rng, n, frames, t):
    s2 = t(rng.uniform(0, 1, (n, 12 * frames)).astype(np.float32))
    r = t(rng.uniform(-1, 1, n).astype(np.float32))
    done = t((rng.uniform(size=n) < 0.3).astype(np.uint8))
    return s2, r, done


def _targets(kind, theta, phi, phi2, frames, r, s2, done, gamma, sd, clip, seed, counter, row_offset, n):
    """y from ss_td3_targets_<kind> (phi2 / sd as given)"""
    L, _l = _lib().lib, _lib()
    y = torch.empty(n, dtype=torch.float32, device="cuda:0")
    c2 = None if phi2 is None else phi2.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    if kind == "f32":
        rc = L.ss_td3_targets_frames(theta.data_ptr(), phi.data_ptr(), c2, frames, r.data_ptr(), s2.data_ptr(), done.data_ptr(), gamma,
                                     sd, clip, seed, counter, row_offset, y.data_ptr(), n, None, 0, st)
    elif kind == "tc":
        ws = torch.empty(_l.td3_tc_workspace_bytes(n), dtype=torch.uint8, device="cuda:0")
        rc = L.ss_td3_targets_tc(theta.data_ptr(), phi.data_ptr(), c2, r.data_ptr(), s2.data_ptr(), done.data_ptr(), gamma, sd, clip,
                                 seed, counter, row_offset, y.data_ptr(), n, ws.data_ptr(), ws.numel(), st)
    else:
        ws = torch.empty(int(L.ss_learner_frames_tc_workspace_bytes(frames, n)), dtype=torch.uint8, device="cuda:0")
        rc = L.ss_td3_targets_frames_tc(theta.data_ptr(), phi.data_ptr(), c2, frames, r.data_ptr(), s2.data_ptr(), done.data_ptr(),
                                        gamma, sd, clip, seed, counter, row_offset, y.data_ptr(), n, ws.data_ptr(), ws.numel(), st)
    assert rc == 0
    return y


def _ddpg(kind, theta, phi, frames, r, s2, done, gamma, n):
    L = _lib().lib
    y = torch.empty(n, dtype=torch.float32, device="cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    if kind == "f32":
        rc = L.ss_ddpg_targets_frames(theta.data_ptr(), phi.data_ptr(), frames, r.data_ptr(), s2.data_ptr(), done.data_ptr(), gamma,
                                      y.data_ptr(), n, st)
    elif kind == "tc":
        ws = torch.empty(8 * n + 64, dtype=torch.uint8, device="cuda:0")
        rc = L.ss_ddpg_targets_tc(theta.data_ptr(), phi.data_ptr(), r.data_ptr(), s2.data_ptr(), done.data_ptr(), gamma, y.data_ptr(),
                                  n, ws.data_ptr(), ws.numel(), st)
    else:
        ws = torch.empty(int(L.ss_learner_frames_tc_workspace_bytes(frames, n)), dtype=torch.uint8, device="cuda:0")
        rc = L.ss_ddpg_targets_frames_tc(theta.data_ptr(), phi.data_ptr(), frames, r.data_ptr(), s2.data_ptr(), done.data_ptr(), gamma,
                                         y.data_ptr(), n, ws.data_ptr(), ws.numel(), st)
    assert rc == 0
    return y


@gpu
@pytest.mark.parametrize("kind,frames", [("f32", 1), ("f32", 4), ("f32", 20), ("tc", 1), ("frames_tc", 4), ("frames_tc", 20)])
def test_one_critic_without_smoothing_is_the_ddpg_target_bit_for_bit(kind, frames):
    rng, theta, phi, _, t = _nets(frames)
    n = 1000
    s2, r, done = _batch(rng, n, frames, t)
    th, ph = t(theta), t(phi)
    want = _ddpg(kind, th, ph, frames, r, s2, done, 0.99, n)
    got = _targets(kind, th, ph, None, frames, r, s2, done, 0.99, 0.0, 0.5, 3, 7, 0, n)
    assert torch.equal(got, want)
    # noise_sd = 0 draws nothing: seed, counter and row offset do not matter
    assert torch.equal(_targets(kind, th, ph, None, frames, r, s2, done, 0.99, 0.0, 0.1, 99, 12345, 4096, n), want)


def _host_eps(n, seed, counter, row_offset=0):
    rows = np.arange(row_offset, row_offset + n, dtype=np.uint64)
    return philox_ref.normal4(seed, _lib().TAG_TARGET_NOISE, rows & np.uint64(0xFFFFFFFF), rows >> np.uint64(32), counter)[:, :2]


@gpu
@pytest.mark.parametrize("frames", [1, 4, 20])
@pytest.mark.parametrize("twin", [False, True])
def test_float32_target_with_smoothing_matches_the_oracle(frames, twin):
    rng, theta, phi, phi2, t = _nets(frames, seed=frames)
    n, seed, counter, off = 777, 11, 5, 3000
    s2, r, done = _batch(rng, n, frames, t)
    y = _targets("f32", t(theta), t(phi), t(phi2) if twin else None, frames, r, s2, done, 0.99, 0.2, 0.5, seed, counter, off, n)
    want = td3_oracle.td3_targets(theta, phi, phi2 if twin else None, r.cpu().numpy(), s2.cpu().numpy(), done.cpu().numpy(), 0.99,
                          _host_eps(n, seed, counter, off), 0.2, 0.5)
    scale = np.abs(want).max()
    assert np.abs(y.cpu().numpy() - want).max() <= 2e-5 * scale
    # the draw matters: without smoothing the target is another one
    y0 = _targets("f32", t(theta), t(phi), t(phi2) if twin else None, frames, r, s2, done, 0.99, 0.0, 0.5, seed, counter, off, n)
    assert not torch.equal(y, y0)


@gpu
@pytest.mark.parametrize("kind,frames", [("tc", 1), ("frames_tc", 4), ("frames_tc", 20)])
@pytest.mark.parametrize("twin", [False, True])
def test_tensor_core_targets_follow_the_float32_target(kind, frames, twin):
    rng, theta, phi, phi2, t = _nets(frames, seed=frames + 1)
    n = 4099
    s2, r, done = _batch(rng, n, frames, t)
    args = (t(theta), t(phi), t(phi2) if twin else None, frames, r, s2, done, 0.99, 0.2, 0.5, 21, 9, 128, n)
    want = _targets("f32", *args).cpu().numpy()
    got = _targets(kind, *args).cpu().numpy()
    assert np.abs(got - want).max() <= 2e-2 * np.abs(want).max()


@gpu
def test_smoothing_noise_statistics():
    """1e6 rows through ss_td3_targets_frames with a zero actor and a critic whose Q is the first action component: gamma = 1,
    reward 0, so y = a~_0 = clamp(clamp(sd eps, -c, c), -1, 1).  Mean 0, the clipped normal's standard deviation, no value
    beyond c; and with a saturated actor every action stays in [-1, 1]."""
    from skillshot_learning_b200.learner import A_N, C_N
    from scipy.stats import norm
    n, sd, c = 1 << 20, 0.2, 0.3
    dev = "cuda:0"
    theta = torch.zeros(A_N, device=dev)
    phi = torch.zeros(C_N, device=dev)
    w = lo.split(phi, lo.critic_shapes(1))
    w[2][256, 0] = 1.0                      # hidden unit 0 = relu(a0), unit 1 = relu(-a0): q = h0 - h1 = a0
    w[2][256, 1] = -1.0
    w[4][0, 0], w[4][1, 0] = 1.0, -1.0
    s2 = torch.zeros((n, 12), device=dev)
    r = torch.zeros(n, device=dev)
    done = torch.zeros(n, dtype=torch.uint8, device=dev)
    y = _targets("f32", theta, phi, None, 1, r, s2, done, 1.0, sd, c, 5, 1, 0, n).double().cpu().numpy()
    assert np.abs(y).max() <= c + 1e-7 and np.abs(y).max() > 0.99 * c
    k = c / sd                             # std of N(0, sd) clipped to [-c, c]
    var = sd * sd * ((1 - 2 * norm.sf(k)) - 2 * k * norm.pdf(k)) + 2 * c * c * norm.sf(k)
    assert abs(y.mean()) < 5 * np.sqrt(var / n)
    assert abs(y.std() - np.sqrt(var)) < 0.005 * np.sqrt(var)
    # every target action in [-1, 1]: an actor saturated at +1 (b3 large) plus noise up to c
    wa = lo.split(theta, lo.actor_shapes(1))
    wa[5][0] = 50.0
    y = _targets("f32", theta, phi, None, 1, r, s2, done, 1.0, 1.0, 0.5, 5, 2, 0, n).cpu().numpy()
    assert y.max() <= 1.0 and y.min() >= 0.5 and (y == 1.0).mean() > 0.4


def _trainer(**kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    base = dict(device="cuda:0", seed=3, batch_size=512, gamma=0.99, tau=0.005, reward_mode="terminal", tick_limit=60)
    base.update(kw)
    return SelfPlayTrainer(base.pop("n_envs", 256), **base)


def _same_state(a, b):
    na, nb = a.networks, b.networks
    for k in ("params", "target", "adam_m", "adam_v"):
        assert torch.equal(getattr(na, k), getattr(nb, k)), k
    assert (na.step_actor, na.step_critic, na.counter) == (nb.step_actor, nb.step_critic, nb.counter)
    for k in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, k), getattr(b.replay, k)), k
    assert (a.replay.pos, a.replay.size, a.replay.counter) == (b.replay.pos, b.replay.size, b.replay.counter)


@gpu
@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_default_td3_options_are_the_ddpg_update(precision, monkeypatch):
    lib = _lib().lib
    calls = []
    real = lib.ss_ddpg_update
    monkeypatch.setattr(lib, "ss_ddpg_update", lambda *a: calls.append(1) or real(*a))
    a = _trainer(precision=precision)
    b = _trainer(precision=precision, twin_critics=False, policy_delay=1, target_noise=0.0, target_noise_clip=0.5)
    assert not b.networks.td3 and a.networks.params.numel() == b.networks.params.numel()
    for _ in range(20):
        for t in (a, b):
            t.rollout(2)
            t.update()
    assert len(calls) == 40
    _same_state(a, b)
    assert set(b.networks.state_dict()) == set(a.networks.state_dict())


@gpu
def test_td3_trainer_rolls_out_as_the_ddpg_trainer():
    """same seed, same actor and critic 1: the rollout does not depend on the TD3 options, only the update does"""
    a = _trainer()
    b = _trainer(twin_critics=True, policy_delay=2, target_noise=0.2)
    assert torch.equal(a.networks.actor, b.networks.actor) and torch.equal(a.networks.critic, b.networks.critic)
    assert not torch.equal(b.networks.critic, b.networks.critic2)
    for _ in range(3):
        a.rollout(4)
        b.rollout(4)
    for k in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, k), getattr(b.replay, k)), k
    assert torch.equal(a.envs.state, b.envs.state) and a.networks.counter == b.networks.counter


@gpu
@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_delayed_updates_leave_actor_and_targets_untouched(precision):
    t = _trainer(precision=precision, twin_critics=True, policy_delay=3, target_noise=0.2)
    net = t.networks
    t.rollout(8)
    views = ("actor", "target_actor", "target_critic", "target_critic2")
    for u in range(1, 10):
        before = {v: getattr(net, v).clone() for v in views + ("critic", "critic2")}
        t.update()
        assert not torch.equal(net.critic, before["critic"]) and not torch.equal(net.critic2, before["critic2"])
        for v in views:
            assert torch.equal(getattr(net, v), before[v]) == (u % 3 != 0), (u, v)
    assert net.step_actor == 3 and net.step_critic == net.step_critic2 == 9 and net.td3_updates == 9
    assert float(net.critic2_sse) > 0


@gpu
@pytest.mark.parametrize("cfg", ["f1", "f20", "pool"])
def test_td3_checkpoint_resumes_mid_cycle(cfg, tmp_path):
    kw = dict(twin_critics=True, policy_delay=3, target_noise=0.2, target_noise_clip=0.5)
    if cfg == "f20":
        kw.update(frames=20, update_precision="bf16", precision="bf16")
    if cfg == "pool":
        from skillshot_learning_b200.learner import A_N
        rng = np.random.default_rng(1)
        kw.update(frames=20, precision="bf16", opponents=[lo.init_actor(rng), lo.init_actor(rng, 20)], pool_envs=128)
    a = _trainer(**kw)
    for _ in range(4):
        a.rollout(2)
        a.update()
    assert a.networks.td3_updates % 3 != 0                    # in the middle of a delay cycle
    a.save(str(tmp_path / "ck.pt"))
    b = _trainer(**kw)
    b.load(str(tmp_path / "ck.pt"))
    for _ in range(5):                                        # across a delayed update
        for t in (a, b):
            t.rollout(2)
            t.update()
    _same_state(a, b)
    assert a.networks.step_critic2 == b.networks.step_critic2 and a.networks.td3_updates == b.networks.td3_updates == 9
    # the refusals on a real trainer, before anything is loaded
    c = _trainer(**dict(kw, twin_critics=False))
    obs = c.obs.clone()
    with pytest.raises(ValueError):
        c.load(str(tmp_path / "ck.pt"))
    assert torch.equal(c.obs, obs)


@gpu
@pytest.mark.parametrize("frames", [1, 20])
def test_six_td3_updates_track_the_oracle(frames):
    """twin critics, delay 2, sd 0.2, c 0.5, Philox dropout, float32: ActorCritic.td3_step against TD3Oracle fed the same
    draws (the smoothing normals of counter k, the two critics' masks of counters k + 1 and k + 2)."""
    from skillshot_learning_b200 import ActorCritic
    rng, theta, phi, _, t = _nets(frames, seed=4)
    ac = ActorCritic(device="cuda:0", seed=7, frames=frames, gamma=0.99, tau=0.005, twin_critics=True, policy_delay=2,
                     target_noise=0.2, target_noise_clip=0.5)
    ac.set_weights(theta, phi, critic2=ac.critic2.clone())
    phi2 = ac.critic2.cpu().numpy()
    orc = td3_oracle.TD3Oracle(theta, phi, phi2, gamma=0.99, tau=0.005, policy_delay=2, sigma=0.2, clip=0.5, dropout=0.2)
    n = 96
    for _ in range(6):
        s = rng.uniform(0, 1, (n, 12 * frames)).astype(np.float32)
        a = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
        s2, r, done = _batch(rng, n, frames, t)
        k = ac.counter
        eps = _host_eps(n, ac.seed, k)
        keep1, keep2 = (philox_ref.dropout_keep(n, ac.seed, k + j, 0.2).astype(np.float32) for j in (1, 2))
        ac.td3_step(t(s), t(a), r, s2, done)
        orc.update(s, a, r.cpu().numpy(), s2.cpu().numpy(), done.cpu().numpy(), eps, keep1, keep2)
        assert ac.counter == k + 3
    for got, want in ((ac.actor, orc.theta), (ac.critic, orc.phi), (ac.critic2, orc.phi2), (ac.target_actor, orc.theta_t),
                      (ac.target_critic, orc.phi_t), (ac.target_critic2, orc.phi2_t)):
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=2e-5)
    assert ac.step_actor == 3 and ac.step_critic == ac.step_critic2 == 6
    assert [len(w) for w in ac.get_weights("critic2")] == [len(w) for w in ac.get_weights("critic")]
