"""GPU parity of the learner kernels (through the C ABI) with the CPU oracle
(oracle/learner_oracle.py; parity unpinned -- see its header) on identical seeded
inputs, every random choice injected or re-derived with tests/philox_ref.py.

Tolerances (float32 kernels against a float32/float64 restatement, different
summation order): forward values 2e-5 relative, gradients 2e-4 relative to the
gradient's scale, parameters after k Adam steps 1e-5 absolute (Adam normalises
the step to ~lr = 1e-3, so this is 1 % of one step)."""
import os

import numpy as np
import pytest
import torch

from oracle import learner_oracle as lo
from tests import philox_ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def net():
    from skillshot_learning_b200 import ActorCritic
    ac = ActorCritic(device="cuda:0", seed=11)
    rng = np.random.default_rng(5)
    theta, phi = lo.init_actor(rng), lo.init_critic(rng)
    # non-zero biases so that every term of the backward pass is exercised
    theta[3072:3328] = rng.normal(0, 0.05, 256); theta[36096:36224] = rng.normal(0, 0.05, 128)
    theta[36480:] = rng.normal(0, 0.05, 2)
    phi[3072:3328] = rng.normal(0, 0.05, 256); phi[36352:36480] = rng.normal(0, 0.05, 128); phi[36608] = 0.1
    ac.set_weights(theta, phi)
    return ac, theta, phi


def _batch(n, seed=0):
    rng = np.random.default_rng(seed)
    s = rng.uniform(0, 1, (n, 12)).astype(np.float32)
    s[:, 4] *= 9.8; s[:, 9] *= 9.8; s[:, 11] = rng.integers(0, 2, n)      # ranges of prepare_states
    a = np.tanh(rng.normal(size=(n, 2))).astype(np.float32)
    r = (-rng.uniform(0, 1, n)).astype(np.float32)
    return s, a, r


def _scale_close(got, want, rel):
    scale = np.abs(want).max() + 1e-12
    np.testing.assert_allclose(got / scale, want / scale, rtol=0, atol=rel)


@pytest.mark.parametrize("n", [1, 16, 33, 1000, 40000])
def test_actor_and_critic_forward(net, n):
    ac, theta, phi = net
    s, a, _ = _batch(n, n)
    got = ac.actor_forward(s).cpu().numpy()
    np.testing.assert_allclose(got, lo.actor_forward(theta, s), rtol=2e-5, atol=2e-6)
    q = ac.critic_forward(s, a).cpu().numpy()
    np.testing.assert_allclose(q, lo.critic_forward(phi, s, a), rtol=2e-5, atol=2e-6)


def test_param_noise_vector_matches_the_host_philox(net):
    ac, theta, _ = net
    for group, counter in ((0, 0), (3, 7), (123456, 2 ** 33 + 5)):
        got = ac.noisy_actor_params(0.5, group=group, counter=counter).cpu().numpy()
        eps = philox_ref.param_noise_eps(lo.ACTOR_PARAMS, ac.seed, group, counter)
        np.testing.assert_allclose(got, lo.noisy_actor_params(theta, eps, 0.5), rtol=1e-5, atol=1e-7)
    eps = philox_ref.param_noise_eps(lo.ACTOR_PARAMS, ac.seed, 0, 0)
    assert abs(eps.mean()) < 0.02 and abs(eps.std() - 1) < 0.02          # N(0,1), SkillshotLearner.py:263


@pytest.mark.parametrize("group", [1, 5, 32, 100])
def test_param_noise_forward_uses_one_draw_per_group(net, group):
    ac, theta, _ = net
    n = 230
    s, _, _ = _batch(n, 77)
    got = ac.actor_forward(s, param_noise_sd=0.5, noise_group=group, counter=9).cpu().numpy()
    want = np.empty_like(got)
    for g in range((n + group - 1) // group):
        eps = philox_ref.param_noise_eps(lo.ACTOR_PARAMS, ac.seed, g, 9)
        sl = slice(g * group, min(n, (g + 1) * group))
        want[sl] = lo.actor_forward(lo.noisy_actor_params(theta, eps, 0.5), s[sl])
    np.testing.assert_allclose(got, want, rtol=5e-5, atol=5e-6)
    again = ac.actor_forward(s, param_noise_sd=0.5, noise_group=group, counter=9).cpu().numpy()
    assert np.array_equal(got, again)                                      # counter-based: reproducible
    other = ac.actor_forward(s, param_noise_sd=0.5, noise_group=group, counter=10).cpu().numpy()
    assert not np.allclose(got, other)


def test_action_noise_distribution(net):
    ac, theta, _ = net
    s, _, _ = _batch(20000, 3)
    clean = ac.actor_forward(s).cpu().numpy()
    noisy = ac.actor_forward(s, action_noise_sd=0.15, counter=4).cpu().numpy()
    d = noisy - clean
    assert abs(d.mean()) < 0.005 and abs(d.std() - 0.15) < 0.005           # N(0, 0.15), SkillshotLearner.py:238
    assert abs(np.corrcoef(d[:, 0], d[:, 1])[0, 1]) < 0.03


@pytest.mark.parametrize("gamma", [0.0, 0.95])
def test_td_targets(net, gamma):
    ac, theta, phi = net
    s2, _, r = _batch(777, 8)
    done = (np.random.default_rng(1).uniform(size=777) < 0.2)
    ac.gamma = gamma
    try:
        y = ac.td_targets(r, s2, torch.from_numpy(done.astype(np.uint8))).cpu().numpy()
    finally:
        ac.gamma = 0.0
    np.testing.assert_allclose(y, lo.ddpg_targets(theta, phi, r, s2, done, gamma), rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize("n", [16, 5, 37, 1000, 20000])
def test_critic_gradient_with_injected_dropout(net, n):
    ac, theta, phi = net
    s, a, r = _batch(n, 100 + n)
    keep = (np.random.default_rng(n).uniform(size=(n, 256)) >= 0.2).astype(np.uint8)
    g = ac.critic_grad(s, a, r, keep=keep).cpu().numpy()
    sse = float(ac.stats[0])
    want, want_sse = lo.critic_grad(phi.astype(np.float64), s, a, r, keep.astype(np.float64), 0.2, dtype=torch.float64)
    _scale_close(g, want, 2e-4)
    assert abs(sse - want_sse) <= 1e-4 * max(1.0, want_sse)
    g2 = ac.critic_grad(s, a, r, keep=keep).cpu().numpy()
    assert np.array_equal(g, g2)                                           # fixed-order reduction


def test_critic_gradient_with_philox_dropout(net):
    ac, theta, phi = net
    n = 300
    s, a, r = _batch(n, 41)
    ac.counter = 1234
    g = ac.critic_grad(s, a, r, row_offset=64).cpu().numpy()
    keep = philox_ref.dropout_keep(n, ac.seed, 1234, 0.2, row_offset=64)
    assert abs(keep.mean() - 0.8) < 0.01                                   # Dropout(0.2), SkillshotLearner.py:105
    want, _ = lo.critic_grad(phi.astype(np.float64), s, a, r, keep.astype(np.float64), 0.2, dtype=torch.float64)
    _scale_close(g, want, 2e-4)


def test_sharded_critic_gradient_sums_to_the_full_batch(net):
    ac, theta, phi = net
    n = 512
    s, a, r = _batch(n, 55)
    keep = (np.random.default_rng(2).uniform(size=(n, 256)) >= 0.2).astype(np.uint8)
    full = ac.critic_grad(s, a, r, keep=keep).cpu().numpy()
    h = n // 2
    parts = [ac.critic_grad(s[i:i + h], a[i:i + h], r[i:i + h], keep=keep[i:i + h], n_global=n).cpu().numpy().copy()
             for i in (0, h)]
    _scale_close(parts[0] + parts[1], full, 2e-6)


@pytest.mark.parametrize("n", [16, 7, 45, 3000])
def test_actor_policy_gradient(net, n):
    ac, theta, phi = net
    s, _, _ = _batch(n, 200 + n)
    g = ac.actor_grad(s).cpu().numpy()
    qsum = float(ac.stats[1])
    want, want_q = lo.actor_grad(theta.astype(np.float64), phi.astype(np.float64), s, dtype=torch.float64)
    _scale_close(g, want, 2e-4)
    assert abs(qsum - want_q) <= 1e-4 * max(1.0, abs(want_q))


def test_adam_and_soft_update(net):
    from skillshot_learning_b200 import ActorCritic
    ac0, theta, phi = net
    ac = ActorCritic(device="cuda:0", seed=1, tau=0.25)
    ac.set_weights(theta, phi)
    opt = lo.AdamTF(lo.CRITIC_PARAMS)
    p, tgt = phi.copy(), phi.copy()
    rng = np.random.default_rng(0)
    for _ in range(5):
        g = rng.normal(0, 0.01, lo.CRITIC_PARAMS).astype(np.float32)
        ac.grads[ac._c_off:].copy_(torch.from_numpy(g))
        ac.apply_adam("critic")
        p = opt.step(p, g)
        tgt = lo.soft_update(tgt, p, 0.25)
    np.testing.assert_allclose(ac.critic.cpu().numpy(), p, rtol=0, atol=2e-6)
    np.testing.assert_allclose(ac.target_critic.cpu().numpy(), tgt, rtol=0, atol=2e-6)
    assert np.array_equal(ac.actor.cpu().numpy(), theta)                   # the other network is untouched


def test_models_fit_tracks_the_reference_learner(net):
    """One episode through models_fit's schedule (SkillshotLearner.py:419-443): critic fitted in
    shuffled batches of 16 (short last batch kept, Dropout on), then the actor stepped on
    consecutive batches; losses and parameters against the oracle with the same orders/masks."""
    from skillshot_learning_b200 import ActorCritic
    _, theta, phi = net
    n, bs = 203, 16
    s, a, r = _batch(n, 999)
    rng = np.random.default_rng(17)
    order = rng.permutation(n)
    keep = (rng.uniform(size=(n, 256)) >= 0.2).astype(np.uint8)
    orc = lo.LearnerOracle(theta, phi, bs)
    want_losses = orc.critic_fit(s, a, r, order, keep.astype(np.float32))
    want_q = orc.actor_fit(s)

    ac = ActorCritic(device="cuda:0", seed=3)
    ac.set_weights(theta, phi)
    ts, ta, tr, tk = (torch.from_numpy(x).cuda() for x in (s, a, r, keep))
    losses, qs = [], []
    for b in range(0, n, bs):
        idx = torch.from_numpy(order[b:b + bs]).cuda()
        sse = ac.critic_step(ts[idx], ta[idx], tr[idx], keep=tk[idx])
        losses.append(float(sse) / len(idx))
    for b in range(0, n, bs):
        qs.append(float(ac.actor_step(ts[b:b + bs])))
    np.testing.assert_allclose(losses, want_losses, rtol=2e-3, atol=1e-6)      # stated tolerance on the losses
    np.testing.assert_allclose(qs, want_q, rtol=2e-3, atol=1e-4)
    np.testing.assert_allclose(ac.critic.cpu().numpy(), orc.phi, rtol=0, atol=1e-5)
    np.testing.assert_allclose(ac.actor.cpu().numpy(), orc.theta, rtol=0, atol=1e-5)
    assert ac.step_critic == 13 and ac.step_actor == 13


def test_replay_ring_push_wrap_and_sample():
    from skillshot_learning_b200 import ReplayRing
    ring = ReplayRing(100, device="cuda:0", seed=5)
    rng = np.random.default_rng(0)
    mirror = dict(obs=np.zeros((100, 12), np.float32), act=np.zeros((100, 2), np.float32), reward=np.zeros(100, np.float32),
                  next_obs=np.zeros((100, 12), np.float32), done=np.zeros(100, np.uint8))
    pos = 0
    for n in (30, 30, 30, 30, 60):                       # wraps twice
        s, a, r = _batch(n, pos + n)
        s2 = rng.uniform(size=(n, 12)).astype(np.float32)
        done_env = rng.integers(0, 2, n // 2).astype(np.uint8)
        ring.push(s, a, r, s2, torch.from_numpy(done_env), done_div=2)
        idx = (pos + np.arange(n)) % 100
        mirror["obs"][idx], mirror["act"][idx], mirror["reward"][idx], mirror["next_obs"][idx] = s, a, r, s2
        mirror["done"][idx] = np.repeat(done_env, 2)
        pos = (pos + n) % 100
    assert ring.pos == pos and ring.size == 100
    for k in mirror:
        assert np.array_equal(getattr(ring, k).cpu().numpy(), mirror[k]), k
    want_idx = rng.integers(0, 100, 64)
    b = ring.sample(64, indices=want_idx)
    for k in mirror:
        assert np.array_equal(b[k].cpu().numpy(), mirror[k][want_idx]), k
    ring.counter = 3
    b = ring.sample(1000)
    idx = b["indices"].cpu().numpy()
    assert np.array_equal(idx, philox_ref.replay_indices(1000, 100, 5, 3))
    assert idx.min() >= 0 and idx.max() < 100 and len(np.unique(idx)) > 90
    assert np.array_equal(b["obs"].cpu().numpy(), mirror["obs"][idx])


def test_reference_surface_trains_one_episode(tmp_path, capsys):
    """SkillshotLearner.main-style use (SkillshotLearner.py:685-693) with a short tick limit."""
    from skillshot_learning_b200 import SkillshotLearner
    skl = SkillshotLearner(device="cuda:0", seed=2)
    skl.save_location = str(tmp_path / "training_models")      # save_boards writes the board rasters there
    skl.model_param_game_tick_limit = 12
    skl.use_random_start = False
    before = skl.networks.actor.clone()
    prog = skl.model_train(epochs=1, save_progress=False, save_boards=True)
    assert prog["epoch_ticks"] == [12] and prog["epoch_winner"] == [0]
    assert len(prog["epoch_board_sequences"][0]) == 12 and prog["epoch_board_sequences"][0][0].shape == (250, 250)
    assert os.path.exists(os.path.join(skl.save_location, "training_boards", "training_boards.npy"))
    assert skl.networks.step_critic == 2 and skl.networks.step_actor == 2      # 24 rows in batches of 16
    assert not torch.equal(before, skl.networks.actor)
    assert np.isfinite(skl.last_fit["critic_loss"])
    state = skl.game_environment.get_state()
    obs = skl.prepare_states([state], 1)[0]
    assert len(obs) == 12
    a = skl.model_act(state, 1)
    assert a.shape == (1, 2) and np.all(np.abs(a) <= 1)


def test_selfplay_trainer_rollout_and_update():
    from skillshot_learning_b200 import SelfPlayTrainer
    tr = SelfPlayTrainer(512, device="cuda:0", seed=4, batch_size=256, noise_group=32, tick_limit=50)
    for _ in range(6):
        out = tr.rollout_tick()
    assert tr.replay.size == 6 * 1024
    # stored transitions chain: next_obs of tick t is obs of tick t+1 for envs that did not reset
    o = tr.replay.obs.cpu().numpy()[:6 * 1024].reshape(6, 1024, 12)
    o2 = tr.replay.next_obs.cpu().numpy()[:6 * 1024].reshape(6, 1024, 12)
    assert np.array_equal(o2[:-1], o[1:])
    r = tr.replay.reward.cpu().numpy()[:1024]
    live = tr.replay.done.cpu().numpy()[:1024] == 0      # a done env was reset: its s' is the fresh game's
    assert live.sum() > 900
    np.testing.assert_allclose(r[live], -o2[0][live, 0] * (353.5533905932738 / 250.0), rtol=2e-5, atol=1e-6)  # looking reward of s'
    before = tr.networks.params.clone()
    sse, q = tr.update()
    assert np.isfinite(float(sse)) and np.isfinite(float(q))
    assert not torch.equal(before, tr.networks.params)


# ---------------------------------------------------------------------------
# tensor-core actor forward (ss_actor_forward_tc)
# ---------------------------------------------------------------------------
def _bf16(x):
    """float32 -> bfloat16 (round to nearest even) -> float32, as cvt.rn.bf16.f32 does."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).reshape(np.shape(x))


def _f16(x):
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float64)


def actor_forward_bf16_model(theta, s):
    """What the tensor-core kernel computes, restated in numpy: layer 1 with fp16 observations and
    fp16 weights, layer 2 with bf16 weights and hidden layer 1 rounded to bf16, fp32 accumulation
    (float64 here), layer 3 and tanh in fp32 (skillshot_learning_b200/csrc/ss_mlp_tc.cu header)."""
    w1, b1, w2, b2, w3, b3 = lo.split(np.asarray(theta, np.float32), lo.ACTOR_SHAPES)
    s = np.asarray(s, np.float32)
    z1 = _f16(s) @ _f16(w1) + b1
    h1 = _bf16(np.maximum(z1, 0).astype(np.float32)).astype(np.float64)
    h2 = np.maximum(h1 @ _bf16(w2).astype(np.float64) + b2, 0)
    return np.tanh(h2 @ w3.astype(np.float64) + b3).astype(np.float32)


@pytest.mark.parametrize("n", [1, 128, 129, 300, 5000, 148 * 128 * 3 + 77])
def test_tensor_core_actor_forward(net, n):
    ac, theta, _ = net
    s, _, _ = _batch(n, 31 + n)
    got = ac.actor_forward(s, precision="bf16").cpu().numpy()
    model = actor_forward_bf16_model(theta, s)
    # against the restated bf16 arithmetic: only fp32 accumulation order and rare 1-ulp flips of
    # the bf16 rounding of a hidden unit differ
    np.testing.assert_allclose(got, model, rtol=0, atol=5e-4)
    # against the exact float32 path: bf16 weight rounding, stated tolerance 2e-2 on actions in [-1, 1]
    np.testing.assert_allclose(got, lo.actor_forward(theta, s), rtol=0, atol=2e-2)


def test_tensor_core_actor_forward_with_noise_groups(net):
    ac, theta, _ = net
    n, group = 1000, 256
    s, _, _ = _batch(n, 78)
    got = ac.actor_forward(s, param_noise_sd=0.5, noise_group=group, action_noise_sd=0.15, counter=21,
                           precision="bf16").cpu().numpy()
    exact = ac.actor_forward(s, param_noise_sd=0.5, noise_group=group, action_noise_sd=0.15, counter=21).cpu().numpy()
    # same Philox draws as the float32 path: the two differ by bf16 rounding only (noisy weights are
    # up to ~3x larger than the clean ones, hence the wider band)
    np.testing.assert_allclose(got, exact, rtol=0, atol=6e-2)
    assert np.abs(got - exact).mean() < 6e-3
    want = np.empty((n, 2), np.float32)
    for g in range((n + group - 1) // group):
        eps = philox_ref.param_noise_eps(lo.ACTOR_PARAMS, ac.seed, g, 21)
        sl = slice(g * group, min(n, (g + 1) * group))
        want[sl] = actor_forward_bf16_model(lo.noisy_actor_params(theta, eps, 0.5), s[sl])
    rows = np.arange(n, dtype=np.uint64)
    zn = philox_ref.normal4(ac.seed, philox_ref.TAG_ACTION_NOISE, rows, np.uint64(0), 21)[:, :2]
    np.testing.assert_allclose(got, want + 0.15 * zn, rtol=0, atol=2e-3)
    with pytest.raises(Exception):
        ac.actor_forward(s, param_noise_sd=0.5, noise_group=100, precision="bf16")    # groups are whole tiles


# ---------------------------------------------------------------------------
# tensor-core critic forward / gradients (ss_critic_forward_tc, ss_critic_grad_tc, ss_actor_grad_tc)
# ---------------------------------------------------------------------------
# Stated tolerances: the operands of every GEMM are bf16 (weights, activations, upstream gradients;
# inputs as hi + lo pairs), accumulation is fp32.  Forward values agree with the float32 path to
# 2e-2 absolute (critic outputs are O(1)), gradients to 2e-2 of the gradient's largest entry
# (typically ~3e-3), after Adam the parameters move by ~lr so they agree to 1e-3 * steps * lr scale.
def _tc_net(net):
    from skillshot_learning_b200 import ActorCritic
    _, theta, phi = net
    ac = ActorCritic(device="cuda:0", seed=11, update_precision="bf16")
    ac.set_weights(theta, phi)
    return ac


@pytest.mark.parametrize("n", [1, 128, 333, 20000])
def test_tensor_core_critic_forward_and_dq_da(net, n):
    ac, theta, phi = net
    s, a, _ = _batch(n, 900 + n)
    q, up = ac.critic_forward(s, a, precision="bf16", want_dq_da=True)
    q, up = q.cpu().numpy(), up.cpu().numpy()
    np.testing.assert_allclose(q, lo.critic_forward(phi, s, a), rtol=0, atol=2e-2)
    at = torch.tensor(a, dtype=torch.float64, requires_grad=True)
    qq = lo.critic_forward_t(torch.tensor(phi, dtype=torch.float64), torch.tensor(s, dtype=torch.float64), at)
    qq.sum().backward()
    # dQ/da sums W3[k] W2[256+m][k] over the ACTIVE hidden units: a unit whose pre-activation sits within
    # bf16 rounding of zero can flip, which moves one row's value by one such term (~5e-3); hence a loose
    # bound on the worst row and a tight one on the average
    want, scale = -at.grad.numpy(), np.abs(at.grad.numpy()).max()
    assert np.abs(up - want).max() <= 0.15 * scale + 5e-3
    assert np.abs(up - want).mean() <= 1e-2 * scale + 5e-4


@pytest.mark.parametrize("n", [1, 128, 333, 20000, 65536 + 77])
def test_actor_and_critic_forward_as_one_launch_equals_the_two_launches(net, n):
    """ss_actor_critic_forward_tc (half of the CTAs play a = actor(s), the other half critic([s, a]), handing each quarter
    tile's actions over through flags) against ss_actor_forward_tc followed by ss_critic_forward_tc: actions, Q, -dQ/da and
    the TD target must be bit-identical; the mailbox comes back empty, so a second call on it works as well."""
    from skillshot_learning_b200._lib import lib, check
    ac = _tc_net(net)
    s, _, r = _batch(n, 7000 + n)
    s = torch.tensor(s, device="cuda"); r = torch.tensor(r, device="cuda")
    done = (torch.arange(n, device="cuda") % 3 == 0).to(torch.uint8)
    a_ref = ac.actor_forward(s, precision="bf16")
    q_ref, up_ref = ac.critic_forward(s, a_ref, precision="bf16", want_dq_da=True)
    y_ref = torch.empty(n, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    check(lib.ss_critic_forward_tc(ac.critic.data_ptr(), s.data_ptr(), a_ref.data_ptr(), n, None, None, r.data_ptr(), done.data_ptr(),
                                   0.9, y_ref.data_ptr(), st), "critic")
    from skillshot_learning_b200 import _lib
    mail = torch.full((n, 2), _lib.PAIR_MAIL_EMPTY, dtype=torch.int32, device="cuda")
    for rep in range(2):
        a = torch.full((n, 2), 7.0, device="cuda"); q = torch.empty(n, device="cuda"); up = torch.empty((n, 2), device="cuda")
        y = torch.empty(n, device="cuda")
        check(lib.ss_actor_critic_forward_tc(ac.actor.data_ptr(), ac.critic.data_ptr(), s.data_ptr(), a.data_ptr(), n, q.data_ptr(),
                                             up.data_ptr(), r.data_ptr(), done.data_ptr(), 0.9, y.data_ptr(), mail.data_ptr(), st),
              "pair")
        torch.cuda.synchronize()
        assert torch.equal(a, a_ref) and torch.equal(q, q_ref) and torch.equal(up, up_ref) and torch.equal(y, y_ref), rep
        assert bool((mail == _lib.PAIR_MAIL_EMPTY).all())


@pytest.mark.parametrize("n", [128, 77, 1000, 20000])
def test_tensor_core_critic_gradient(net, n):
    ac = _tc_net(net)
    _, theta, phi = net
    s, a, r = _batch(n, 300 + n)
    keep = (np.random.default_rng(n).uniform(size=(n, 256)) >= 0.2).astype(np.uint8)
    g = ac.critic_grad(s, a, r, keep=keep).cpu().numpy()
    sse = float(ac.stats[0])
    want, want_sse = lo.critic_grad(phi.astype(np.float64), s, a, r, keep.astype(np.float64), 0.2, dtype=torch.float64)
    _scale_close(g, want, 2e-2)
    assert np.abs(g - want).mean() < 2e-3 * np.abs(want).max()
    assert abs(sse - want_sse) <= 2e-2 * max(1.0, want_sse)
    again = ac.critic_grad(s, a, r, keep=keep).cpu().numpy()
    assert np.array_equal(g, again)


def test_tensor_core_critic_gradient_philox_dropout_matches_float32_path(net):
    ac = _tc_net(net)
    ac32, theta, phi = net
    n = 1000
    s, a, r = _batch(n, 42)
    ac.counter = ac32.counter = 77
    ac.seed = ac32.seed
    g = ac.critic_grad(s, a, r, row_offset=5).cpu().numpy()
    ac32.counter = 77
    want = ac32.critic_grad(s, a, r, row_offset=5).cpu().numpy()      # same Philox mask in both kernels
    _scale_close(g, want, 2e-2)


@pytest.mark.parametrize("n", [128, 45, 3000, 20000])
def test_tensor_core_actor_policy_gradient(net, n):
    ac = _tc_net(net)
    _, theta, phi = net
    s, _, _ = _batch(n, 500 + n)
    g = ac.actor_grad(s).cpu().numpy()
    qsum = float(ac.stats[1])
    want, want_q = lo.actor_grad(theta.astype(np.float64), phi.astype(np.float64), s, dtype=torch.float64)
    _scale_close(g, want, 2e-2)
    assert np.abs(g - want).mean() < 2e-3 * np.abs(want).max()
    assert abs(qsum - want_q) <= 2e-2 * max(1.0, abs(want_q))


def test_tensor_core_td_targets(net):
    ac = _tc_net(net)
    _, theta, phi = net
    s2, _, r = _batch(3000, 8)
    done = (np.random.default_rng(1).uniform(size=3000) < 0.2)
    ac.gamma = 0.95
    y = ac.td_targets(r, s2, torch.from_numpy(done.astype(np.uint8))).cpu().numpy()
    np.testing.assert_allclose(y, lo.ddpg_targets(theta, phi, r, s2, done, 0.95), rtol=0, atol=2e-2)
    assert np.array_equal(y[done], r[done])


def test_tensor_core_update_tracks_the_float32_update(net):
    """Twenty DDPG updates of 4,096 rows with the tensor-core kernels against the same updates with the
    float32 kernels (same batches, injected masks): the losses track, the parameters stay close."""
    from skillshot_learning_b200 import ActorCritic
    _, theta, phi = net
    nets = [ActorCritic(device="cuda:0", seed=1, gamma=0.9, tau=0.05, update_precision=p) for p in ("f32", "bf16")]
    for ac in nets:
        ac.set_weights(theta, phi)
    rng = np.random.default_rng(3)
    losses = [[], []]
    for it in range(20):
        s, a, r = _batch(4096, 7000 + it)
        s2, _, _ = _batch(4096, 8000 + it)
        keep = torch.from_numpy((rng.uniform(size=(4096, 256)) >= 0.2).astype(np.uint8)).cuda()
        for k, ac in enumerate(nets):
            y = ac.td_targets(r, s2)
            losses[k].append(float(ac.critic_step(s, a, y, keep=keep)) / 4096)
            ac.actor_step(s)
    np.testing.assert_allclose(losses[1], losses[0], rtol=3e-2, atol=1e-4)
    d = (nets[0].params - nets[1].params).abs()
    assert float(d.max()) < 20 * 1e-3 * 0.5 and float(d.mean()) < 1e-3          # a fraction of the distance moved


@pytest.mark.parametrize("capacity", [2048 * 8, 2048 * 8 + 100])
def test_library_side_rollout_loop_equals_per_tick_calls(capacity):
    """ss_selfplay_rollout (n ticks enqueued by one call) against n rollout_tick calls: same kernels, same Philox
    counters -> identical env state, observations and replay rows.  With a ring that is a whole number of ticks the
    library produces the transitions in place in the ring (no copy kernel); otherwise it pushes them tick by tick."""
    from skillshot_learning_b200 import SelfPlayTrainer
    trs = [SelfPlayTrainer(1024, device="cuda:0", seed=9, batch_size=256, noise_group=128, tick_limit=30, precision=p,
                           replay_capacity=capacity) for p in ("f32", "f32", "bf16", "bf16")]
    for k in (0, 2):
        for _ in range(7):
            trs[k].rollout_tick()
        trs[k + 1].rollout(4)
        trs[k + 1].rollout(3)
        a, b = trs[k], trs[k + 1]
        assert a.replay.size == b.replay.size == 7 * 2048 and a.replay.pos == b.replay.pos
        for name in ("obs", "act", "reward", "next_obs", "done"):
            assert torch.equal(getattr(a.replay, name), getattr(b.replay, name)), name
        assert torch.equal(a.obs, b.obs) and torch.equal(a.envs.state, b.envs.state)
        assert torch.equal(a.actions, b.actions)
        assert a.envs.counter == b.envs.counter and a.networks.counter == b.networks.counter
        b.rollout(12)                                      # wraps the ring
        for _ in range(12):
            a.rollout_tick()
        for name in ("obs", "act", "reward", "next_obs", "done"):
            assert torch.equal(getattr(a.replay, name), getattr(b.replay, name)), name
        assert torch.equal(a.obs, b.obs) and a.replay.pos == b.replay.pos and a.replay.size == b.replay.size


def test_overlapped_rollout_equals_the_two_kernel_rollout(monkeypatch):
    """SS_ROLLOUT_OVERLAP=1 (ss_selfplay_rollout2: the env step consumes the forward kernel's action tiles while that kernel
    is still running, on a second stream) against the default back-to-back kernels at a size where both grids are resident
    together: identical replay rows, observations, env state and counters; the tile counters are handed back zeroed."""
    from skillshot_learning_b200 import SelfPlayTrainer
    mk = lambda: SelfPlayTrainer(1024, device="cuda:0", seed=9, batch_size=256, noise_group=128, tick_limit=30, precision="bf16",
                                 replay_capacity=2048 * 8)
    a = mk()
    a.rollout(4); a.rollout(3); a.rollout(12)
    monkeypatch.setenv("SS_ROLLOUT_OVERLAP", "1")
    b = mk()
    b.rollout(4); b.rollout(3); b.rollout(12)
    torch.cuda.synchronize()
    assert b._tile_ready is not None and int(b._tile_ready.abs().sum()) == 0
    b.envs.check_status()
    for name in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, name), getattr(b.replay, name)), name
    assert torch.equal(a.obs, b.obs) and torch.equal(a.envs.state, b.envs.state) and torch.equal(a.actions, b.actions)
    assert a.replay.pos == b.replay.pos and a.envs.counter == b.envs.counter and a.networks.counter == b.networks.counter


def test_chained_launches_and_forward_pairs_change_no_bit(monkeypatch):
    """The rollout and the update as dependent-launch chains with the actor -> critic forward pairs as one launch each (the
    default) against ordinary launches and separate forward kernels: after interleaved rollouts and updates every
    parameter, Adam moment, target, replay row and env state must be bit-identical."""
    from skillshot_learning_b200 import SelfPlayTrainer
    from skillshot_learning_b200._lib import lib
    mk = lambda: SelfPlayTrainer(4096, device="cuda:0", seed=21, batch_size=8192 + 77, noise_group=256, tick_limit=40, precision="bf16",
                                 replay_capacity=8192 * 6, gamma=0.97, tau=0.01)
    def run(tr):
        for _ in range(6):
            tr.rollout(3)
            tr.update(); tr.update()
        torch.cuda.synchronize()
        return tr
    a = run(mk())                                                   # default: chained, paired
    assert a.networks._pair_mail is not None
    prev = lib.ss_set_dependent_launch(0)
    monkeypatch.setenv("SS_UPDATE_PAIR", "0")
    try:
        b = run(mk())
    finally:
        lib.ss_set_dependent_launch(prev)
    assert b.networks._pair_mail is None
    for name in ("params", "target", "adam_m", "adam_v"):
        assert torch.equal(getattr(a.networks, name), getattr(b.networks, name)), name
    for name in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, name), getattr(b.replay, name)), name
    assert torch.equal(a.envs.state, b.envs.state) and torch.equal(a.obs, b.obs)
    assert bool((a.networks._pair_mail == _pair_empty()).all())
    a.envs.check_status()


def _pair_empty():
    from skillshot_learning_b200 import _lib
    return _lib.PAIR_MAIL_EMPTY


def test_fused_forward_and_env_step_kernel_equals_the_two_kernels():
    """ss_actor_forward_step_tc (the rollout tick as ONE kernel: the env step of a row is played in the forward kernel's
    output stage by the lane that computed its action; off by default in ss_selfplay_rollout because it is slower) against
    ss_actor_forward_tc followed by the env step: actions, next observations, rewards, flags, episode statistics and the env
    state must be bit-identical, tick after tick, through hits, tick-limit restarts and parameter noise."""
    from skillshot_learning_b200 import ActorCritic, SkillshotEnvs, _lib
    from skillshot_learning_b200._lib import lib, check
    n = 1000                                                        # rows 2,000: a ragged last tile
    ac = ActorCritic(device="cuda:0", seed=3)
    a_envs, b_envs = (SkillshotEnvs(n, device="cuda:0", random_positions=True, seed=5, reward_mode="looking", tick_limit=12,
                                    auto_reset=True) for _ in range(2))
    for e in (a_envs, b_envs):
        e.collect_episode_stats = True
    obs_a = a_envs.observe().contiguous()
    obs_b = obs_a.clone()
    act_a, act_b = (torch.empty((n, 2, 2), device="cuda") for _ in range(2))
    nxt = torch.empty((n, 2, 12), device="cuda"); nxt2 = torch.empty_like(nxt)
    rew = torch.empty((n, 2), device="cuda"); done = torch.empty(n, dtype=torch.uint8, device="cuda")
    win = torch.empty_like(done); rows = torch.empty((n, 2), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    restarts = 0
    for t in range(40):
        # two kernels
        ac.actor_forward(obs_a.view(-1, 12), param_noise_sd=0.5, noise_group=256, out=act_a.view(-1, 2), counter=t, precision="bf16")
        out = a_envs.step(act_a, obs_out=obs_a)
        # one kernel
        check(lib.ss_actor_forward_step_tc(ac.actor.data_ptr(), obs_b.data_ptr(), act_b.data_ptr(), 2 * n, 0.5, 256, 0.0, ac.seed, t,
                                           b_envs.state.data_ptr(), nxt.data_ptr(), nxt2.data_ptr(), rew.data_ptr(), done.data_ptr(),
                                           rows.data_ptr(), win.data_ptr(), _lib.REWARD_LOOKING, 12, _lib.RESET_RANDOM, b_envs.seed,
                                           b_envs.counter, b_envs.status.data_ptr(), _lib.STEP_EPISODE_STATS, st), "fused")
        b_envs.counter += 1
        assert torch.equal(act_a, act_b), t
        assert torch.equal(obs_a, nxt) and torch.equal(nxt, nxt2), t
        assert torch.equal(out["reward"], rew) and torch.equal(out["done"], done) and torch.equal(out["winner"], win), t
        assert torch.equal(rows, (win != 0).to(torch.uint8)[:, None].expand(n, 2)), t
        assert torch.equal(a_envs.state, b_envs.state), t
        restarts += int(done.sum())
        obs_b.copy_(nxt)
    assert restarts > 2 * n
    sa, sb = a_envs.episode_summary(), b_envs.episode_summary()
    assert sa["episodes"] == sb["episodes"] == restarts and np.array_equal(sa["histogram"], sb["histogram"])
    b_envs.check_status()


@pytest.mark.parametrize("precision,gamma,tau", [("f32", 0.0, 1.0), ("f32", 0.97, 0.01), ("bf16", 0.97, 0.01)])
def test_single_call_update_equals_the_stepwise_update(precision, gamma, tau):
    """ss_ddpg_update (the whole update enqueued by one host call) against sample / target / critic step /
    actor step called one by one: same kernels, same arguments, same Philox counters -> identical weights,
    optimiser state, targets, gradients, statistics and minibatch."""
    from skillshot_learning_b200 import SelfPlayTrainer
    a, b = [SelfPlayTrainer(1024, device="cuda:0", seed=5, batch_size=3000, noise_group=128, tick_limit=30, precision=precision,
                            gamma=gamma, tau=tau) for _ in range(2)]
    for tr in (a, b):
        tr.rollout(5)
    for it in range(4):
        sa, qa = a.update()
        sb, qb = b.update_stepwise()
        assert float(sa) == float(sb) and float(qa) == float(qb), it
        na, nb = a.networks, b.networks
        for name in ("params", "target", "adam_m", "adam_v", "grads"):
            assert torch.equal(getattr(na, name), getattr(nb, name)), (it, name)
        for name in ("obs", "act", "reward", "next_obs", "done", "indices"):
            assert torch.equal(a._batch[name], b._batch[name]), (it, name)
        assert (na.counter, na.step_actor, na.step_critic, a.replay.counter) == (nb.counter, nb.step_actor, nb.step_critic, b.replay.counter)
    assert not torch.equal(a.networks.params, SelfPlayTrainer(8, device="cuda:0", seed=5).networks.params)


def test_reference_surface_persistence_round_trip(tmp_path, capsys):
    """save / load of models, progress CSV and board rasters in the reference's directory layout
    (SkillshotLearner.py:123-204), plus the full optimiser / Philox state for resuming."""
    from skillshot_learning_b200 import SkillshotLearner
    skl = SkillshotLearner(device="cuda:0", seed=3)
    skl.save_location = str(tmp_path / "training_models")
    skl.model_param_game_tick_limit = 6
    skl.use_random_start = False
    skl.model_train(epochs=2, save_progress=True, save_boards=True)
    assert sorted(os.listdir(os.path.join(skl.save_location, "actor"))) == ["0_2_model.npz"]
    prog = skl.load_training_progress()
    assert list(prog["epoch_ticks"]) == [6, 6] and list(prog["epoch_winner"]) == [0, 0]
    boards = skl.load_training_boards()
    assert len(boards) == 2 and boards[0].shape == (6, 250, 250)
    skl.model_train(epochs=1, save_progress=True, save_boards=False)
    assert sorted(os.listdir(os.path.join(skl.save_location, "critic"))) == ["0_2_model.npz", "3_4_model.npz"]
    assert len(skl.load_training_progress()) == 3
    first = {k: v.copy() for k, v in np.load(os.path.join(skl.save_location, "actor", "0_2_model.npz")).items()}
    other = SkillshotLearner(device="cuda:0", seed=99)
    other.save_location = skl.save_location
    assert other.load_actor_critic_models() is True              # SkillshotLearner.py:123-137 returns True / False
    assert torch.equal(other.networks.params, skl.networks.params)
    assert torch.equal(other.networks.adam_m, skl.networks.adam_m) and other.networks.step_critic == skl.networks.step_critic
    state = skl.game_environment.get_state()
    assert np.array_equal(other.model_act(state, 1), skl.model_act(state, 1))
    # load_index selects the epoch range, weights AND optimiser state: the first save is not the latest one
    steps_latest = other.networks.step_critic
    assert other.load_actor_critic_models(load_index=0) is True
    assert np.array_equal(np.concatenate([w.ravel() for w in other.networks.get_weights("actor")]),
                          np.concatenate([first[k].ravel() for k in first]))
    assert not torch.equal(other.networks.params, skl.networks.params) and 0 < other.networks.step_critic < steps_latest
    # nothing saved: False, like the reference
    empty = SkillshotLearner(device="cuda:0", seed=1)
    empty.save_location = str(tmp_path / "nothing_here")
    assert empty.load_actor_critic_models() is False
    os.makedirs(os.path.join(empty.save_location, "actor"))
    assert empty.load_actor_critic_models() is False


# ---------------------------------------------------------------------------
# BASELINE.json's full sizes (configs 3-4: 524,288 rows per tick / update) through size-independent properties
# ---------------------------------------------------------------------------
def test_full_size_actor_forward_properties(net):
    """524,288 rows: (1) a sample of rows against the oracle, (2) row-permutation equivariance, bit for bit (a row's
    action depends on that row only, whatever tile, CTA or lane it lands in), (3) repeatability."""
    ac, theta, _ = net
    n = 524288
    g = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.rand((n, 12), device="cuda", generator=g)
    obs[:, 4] *= 9.8
    obs[:, 9] *= 9.8
    for precision, tol in (("f32", 2e-5), ("bf16", 2e-2)):
        act = ac.actor_forward(obs, precision=precision)
        idx = torch.randint(0, n, (2000,), device="cuda", generator=g)
        want = lo.actor_forward(theta, obs[idx].cpu().numpy())
        np.testing.assert_allclose(act[idx].cpu().numpy(), want, rtol=0, atol=tol)
        perm = torch.randperm(n, device="cuda", generator=g)
        assert torch.equal(ac.actor_forward(obs[perm].contiguous(), precision=precision), act[perm])
        assert torch.equal(ac.actor_forward(obs, precision=precision), act)


def test_full_size_gradients_are_additive_over_shards(net):
    """524,288 rows: the gradient of the whole batch equals the sum of the gradients of its two halves taken with the
    global divisor (what the multi-GPU update relies on), for both kernel families."""
    from skillshot_learning_b200 import ActorCritic
    _, theta, phi = net
    n = 524288
    g = torch.Generator(device="cuda").manual_seed(6)
    s = torch.rand((n, 12), device="cuda", generator=g)
    a = torch.rand((n, 2), device="cuda", generator=g) * 2 - 1
    y = -torch.rand(n, device="cuda", generator=g)
    for precision, tol in (("bf16", 2e-4), ("f32", 2e-5)):
        ac = ActorCritic(device="cuda:0", seed=13, update_precision=precision)
        ac.set_weights(theta, phi)
        h = n // 2
        ac.counter = 50
        full = ac.critic_grad(s, a, y).clone()
        parts = []
        for k in range(2):
            ac.counter = 50
            parts.append(ac.critic_grad(s[k * h:(k + 1) * h], a[k * h:(k + 1) * h], y[k * h:(k + 1) * h],
                                        n_global=n, row_offset=k * h).clone())
        scale = float(full.abs().max())
        assert float((parts[0] + parts[1] - full).abs().max()) <= tol * scale
        fa = ac.actor_grad(s).clone()
        pa = [ac.actor_grad(s[k * h:(k + 1) * h]).clone() for k in range(2)]
        assert float((pa[0] + pa[1] - fa).abs().max()) <= tol * float(fa.abs().max())
        assert torch.isfinite(full).all() and torch.isfinite(fa).all()


# ---------------------------------------------------------------------------
# frame-stacked planning actor (BASELINE.json configs[4]; no reference code: parity unpinned, reduction tested)
# ---------------------------------------------------------------------------
def test_frame_stack_actor_reduces_to_the_reference_actor(net):
    from skillshot_learning_b200 import FrameStackActor
    ac, theta, _ = net
    n = 333
    fa = FrameStackActor(n, frames=1, device="cuda:0", seed=1)
    assert fa.n_params == lo.ACTOR_PARAMS
    fa.params.copy_(torch.from_numpy(theta).cuda())
    s, _, _ = _batch(n, 12)
    fa.push(s)
    assert torch.equal(fa.forward(), ac.actor_forward(s))                  # frames = 1 IS the reference actor


def test_frame_stack_actor_ring_order_restarts_and_noise_groups():
    from skillshot_learning_b200 import FrameStackActor
    n, F = 301, 20
    fa = FrameStackActor(n, frames=F, device="cuda:0", seed=3)
    assert fa.n_params == 12 * F * 256 + 256 + 256 * 128 + 128 + 128 * 2 + 2
    theta = fa.params.cpu().numpy()
    rng = np.random.default_rng(0)
    hist = np.zeros((n, F, 12), np.float32)                                # mirror, oldest -> newest
    for t in range(27):                                                    # wraps the ring
        s = rng.uniform(0, 1, (n, 12)).astype(np.float32)
        done_env = (rng.uniform(size=(n + 1) // 2) < 0.1).astype(np.uint8)
        restart = np.repeat(done_env, 2)[:n].astype(bool) if t > 0 else np.ones(n, bool)
        fa.push(s, torch.from_numpy(done_env))
        hist = np.concatenate([hist[:, 1:], s[:, None]], axis=1)
        hist[restart] = s[restart][:, None, :]
        np.testing.assert_array_equal(fa.ordered_stack().cpu().numpy(), hist.reshape(n, F * 12))
        if t % 9 == 0:
            got = fa.forward().cpu().numpy()
            np.testing.assert_allclose(got, lo.frames_actor_forward(theta, hist.reshape(n, F * 12), F), rtol=2e-5, atol=2e-6)
    group = 64
    fa.counter = 5
    got = fa.forward(param_noise_sd=0.5, noise_group=group).cpu().numpy()
    x = hist.reshape(n, F * 12)
    for g in range((n + group - 1) // group):
        eps = philox_ref.param_noise_eps(fa.n_params, fa.seed, g, 5)
        sl = slice(g * group, min(n, (g + 1) * group))
        want = lo.frames_actor_forward(lo.noisy_actor_params(theta, eps, 0.5), x[sl], F)
        np.testing.assert_allclose(got[sl], want, rtol=1e-4, atol=1e-5)


def frames_forward_tc_model(theta, x, frames):
    """What ss_actor_forward_frames_tc computes, restated in numpy (ss_frames_tc.cu header): layer 1 with fp16
    inputs and weights, hidden layer 1 rounded to bf16, bf16 W2, fp32 accumulation (float64 here), fp32 output layer."""
    shapes = [(12 * frames, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
    w1, b1, w2, b2, w3, b3 = lo.split(np.asarray(theta, np.float32), shapes)
    z1 = _f16(x) @ _f16(w1) + b1
    h1 = _bf16(np.maximum(z1, 0).astype(np.float32)).astype(np.float64)
    h2 = np.maximum(h1 @ _bf16(w2).astype(np.float64) + b2, 0)
    return np.tanh(h2 @ w3.astype(np.float64) + b3).astype(np.float32)


@pytest.mark.parametrize("frames,n", [(1, 77), (5, 300), (20, 1), (20, 128), (20, 1000), (11, 148 * 128 * 2 + 77)])
def test_tensor_core_frame_stack_actor(frames, n):
    from skillshot_learning_b200 import FrameStackActor
    exact = FrameStackActor(n, frames=frames, device="cuda:0", seed=8)
    fast = FrameStackActor(n, frames=frames, device="cuda:0", seed=8, precision="bf16")
    assert torch.equal(exact.params, fast.params)
    bias = torch.Generator(device="cpu").manual_seed(2)
    with torch.no_grad():                                                  # non-zero biases: they ride through the MMA
        o = 12 * frames * 256
        exact.params[o:o + 256] = (torch.randn(256, generator=bias) * 0.05).cuda()
        exact.params[-2:] = torch.tensor([0.01, -0.02]).cuda()
        fast.params.copy_(exact.params)
    g = torch.Generator(device="cuda").manual_seed(4)
    for t in range(frames + 3):                                            # fills and wraps the ring
        s = torch.rand((n, 12), device="cuda", generator=g)
        s[:, 4] *= 9.87                                                    # the rotation term's range (prepare_states)
        exact.push(s)
        fast.push(s)
    # the tensor-core path keeps its history as fp16 operand tiles: same frames, same order, rounded once
    assert torch.equal(fast.ordered_stack(), exact.ordered_stack().half().float())
    got = fast.forward().cpu().numpy()
    ref = exact.forward().cpu().numpy()
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, ref, rtol=0, atol=3e-2)
    assert np.abs(got - ref).mean() < 3e-3
    rows = np.unique(np.concatenate([np.arange(min(n, 300)), np.arange(max(0, n - 300), n)]))
    x = exact.ordered_stack().cpu().numpy()[rows]
    np.testing.assert_allclose(got[rows], frames_forward_tc_model(fast.params.cpu().numpy(), x, frames), rtol=0, atol=2e-3)


def test_tensor_core_frame_stack_actor_noise_groups():
    from skillshot_learning_b200 import FrameStackActor
    n, F, group = 1500, 20, 256
    exact = FrameStackActor(n, frames=F, device="cuda:0", seed=3)
    fast = FrameStackActor(n, frames=F, device="cuda:0", seed=3, precision="bf16")
    g = torch.Generator(device="cuda").manual_seed(5)
    for t in range(27):                                                    # wraps the ring, with restarts
        s = torch.rand((n, 12), device="cuda", generator=g)
        done = (torch.rand(n // 2, device="cuda", generator=g) < 0.1).to(torch.uint8)
        exact.push(s, done)
        fast.push(s, done)
    assert torch.equal(fast.ordered_stack(), exact.ordered_stack().half().float())
    exact.counter = fast.counter = 9
    ref = exact.forward(param_noise_sd=0.5, noise_group=group).cpu().numpy()
    got = fast.forward(param_noise_sd=0.5, noise_group=group).cpu().numpy()
    np.testing.assert_allclose(got, ref, rtol=0, atol=8e-2)                # same Philox vectors; bf16 / fp16 rounding only
    assert np.abs(got - ref).mean() < 8e-3
    theta, x = fast.params.cpu().numpy(), fast.ordered_stack().cpu().numpy()
    for gi in range((n + group - 1) // group):
        eps = philox_ref.param_noise_eps(fast.n_params, fast.seed, gi, 9)
        sl = slice(gi * group, min(n, (gi + 1) * group))
        want = frames_forward_tc_model(lo.noisy_actor_params(theta, eps, 0.5), x[sl], F)
        np.testing.assert_allclose(got[sl], want, rtol=0, atol=3e-3)
    with pytest.raises(Exception):
        fast.forward(param_noise_sd=0.5, noise_group=100)                  # groups are whole tiles


def test_full_size_frame_stack_actor_is_invariant_to_the_ring_phase():
    """BASELINE.json configs[4] size (131,072 rows x 20 frames).  Two actors see the same last 20 frames but their rings
    are at different phases (one has been pushed 7 more times before): the network input is the same history, so the
    float32 path must give identical actions and the tensor-core path -- which rotates W1's rows instead of the data --
    the same up to the order of its fp32 sums.  Also the tensor-core path against the float32 path at this size."""
    from skillshot_learning_b200 import FrameStackActor
    n, F = 131072, 20
    g = torch.Generator(device="cuda").manual_seed(11)
    outs = {}
    for precision in ("f32", "bf16"):
        a = FrameStackActor(n, frames=F, device="cuda:0", seed=2, precision=precision)
        b = FrameStackActor(n, frames=F, device="cuda:0", seed=2, precision=precision)
        g.manual_seed(11)
        for _ in range(7):
            b.push(torch.rand((n, 12), device="cuda", generator=g))
        for _ in range(F + 4):
            s = torch.rand((n, 12), device="cuda", generator=g)
            a.push(s)
            b.push(s)
        assert a.head % F != b.head % F
        assert torch.equal(a.ordered_stack(), b.ordered_stack())
        oa, ob = a.forward(), b.forward()
        if precision == "f32":
            assert torch.equal(oa, ob)
        else:
            # a different order of the fp32 sums moves a hidden unit across a bf16 rounding boundary now and then
            assert float((oa - ob).abs().max()) < 2e-3 and float((oa - ob).abs().mean()) < 1e-5
        a.counter = b.counter = 3
        na, nb = a.forward(param_noise_sd=0.5, noise_group=1024), b.forward(param_noise_sd=0.5, noise_group=1024)
        assert float((na - nb).abs().max()) < (1e-6 if precision == "f32" else 5e-3)
        assert float((na - nb).abs().mean()) < (1e-7 if precision == "f32" else 5e-5)
        assert torch.isfinite(na).all() and float((na - oa).abs().mean()) > 1e-3          # the noise does something
        outs[precision] = (oa, na)
    for k in range(2):
        d = (outs["bf16"][k] - outs["f32"][k]).abs()
        assert float(d.max()) < (3e-2, 1e-1)[k] and float(d.mean()) < (3e-3, 8e-3)[k]


@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_trainer_checkpoint_resumes_bit_identically(tmp_path, precision):
    """SURVEY.md 8(f) rank 1: a batched run saved and resumed (games in flight, replay ring, weights, Adam moments, targets,
    every Philox counter) continues exactly as the uninterrupted run does."""
    from skillshot_learning_b200 import SelfPlayTrainer
    kw = dict(device="cuda:0", seed=17, batch_size=2000, noise_group=128, tick_limit=25, gamma=0.9, tau=0.05, precision=precision,
              replay_capacity=2048 * 6)
    a = SelfPlayTrainer(1024, **kw)
    for _ in range(3):
        a.rollout(3)
        a.update()
    a.save(str(tmp_path / "ckpt" / "trainer.pt"))
    b = SelfPlayTrainer(1024, **dict(kw, seed=99))                       # different seeds: everything must come from the file
    b.load(str(tmp_path / "ckpt" / "trainer.pt"))
    for tr in (a, b):
        for _ in range(3):
            tr.rollout(4)                                                # wraps the ring
            tr.update()
    for name in ("params", "target", "adam_m", "adam_v", "grads"):
        assert torch.equal(getattr(a.networks, name), getattr(b.networks, name)), name
    for name in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, name), getattr(b.replay, name)), name
    assert torch.equal(a.envs.state, b.envs.state) and torch.equal(a.obs, b.obs)
    assert (a.ticks, a.replay.pos, a.replay.size, a.networks.counter, a.envs.counter) == (
        b.ticks, b.replay.pos, b.replay.size, b.networks.counter, b.envs.counter)


def test_trainer_board_export_and_progress(tmp_path):
    """SURVEY.md 8(f) ranks 2-3 for batched runs: board rasters of one game of the batch for the host display tools, and
    the per-episode log reduced on the device."""
    from skillshot_learning_b200 import SelfPlayTrainer
    tr = SelfPlayTrainer(512, device="cuda:0", seed=2, batch_size=256, noise_group=128, tick_limit=12, replay_capacity=1024 * 40)
    boards = tr.record_boards(7, 30, path=str(tmp_path / "training_boards"))
    assert boards.shape == (30, 250, 250) and set(np.unique(boards)) <= {0, 1, 2, 3, 4}
    st = tr.envs.export_state(7, 1)
    body = np.argwhere(boards[-1] == 1)                                   # player 1's 3 x 3 body sits at pos + 1
    assert body.min(axis=0).tolist() == [int(st["px"][0, 0]) + 1, int(st["py"][0, 0]) + 1] and len(body) >= 8
    saved = np.load(str(tmp_path / "training_boards" / "training_boards.npy"), allow_pickle=True)
    assert saved.shape == (1,) and np.array_equal(saved[0], boards)
    p = tr.progress()
    assert p["episodes"] >= 2 * 512 and p["episodes"] == p["player1_hit"] + p["player2_hit"] + p["tick_limit"]
    assert 1 <= p["mean_ticks"] <= 12 and int(p["histogram"].sum()) == p["episodes"]


@pytest.mark.parametrize("precision", ["f32", "bf16"])
@pytest.mark.parametrize("batch", [1, 127, 129])
def test_single_call_update_at_ragged_batch_sizes(precision, batch):
    """ss_ddpg_update at batch sizes around the 128-row tile (and a single row) against the stepwise update."""
    from skillshot_learning_b200 import SelfPlayTrainer
    a, b = [SelfPlayTrainer(64, device="cuda:0", seed=8, batch_size=batch, noise_group=128, tick_limit=20, precision=precision,
                            gamma=0.9, tau=0.1) for _ in range(2)]
    for tr in (a, b):
        tr.rollout(3)
    for _ in range(3):
        a.update()
        b.update_stepwise()
    for name in ("params", "target", "adam_m", "adam_v", "grads", "stats"):
        assert torch.equal(getattr(a.networks, name), getattr(b.networks, name)), name
    assert torch.isfinite(a.networks.params).all()


def test_peer_exchange_kernels_with_a_world_of_one_equal_the_local_reduction():
    """The exchange kernels on a single GPU (world = 1: the rank pushes into its own inbox and waits for its own flag):
    ss_peer_reduce_push + ss_peer_adam_tf, and the one-kernel form ss_peer_reduce_adam_tf, must leave exactly the parameters,
    Adam moments, target, summed gradient and extra-slot sum that ss_reduce_adam_tf leaves, over several epochs (both inbox
    parities).  (The multi-GPU behaviour is covered by tests/test_gpu_multi.py and bench.py's peer_check.)"""
    import ctypes
    from skillshot_learning_b200._lib import lib, check
    n, parts = 36609, 37
    st = torch.cuda.current_stream().cuda_stream
    own = ctypes.c_void_p()
    check(lib.ss_peer_alloc(1, n, ctypes.byref(own)), "alloc")
    try:
        bases = (ctypes.c_void_p * 1)(own.value)
        g = torch.Generator(device="cuda"); g.manual_seed(3)
        mk = lambda: dict(p=torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)),
                          m=torch.zeros(n, device="cuda"), v=torch.zeros(n, device="cuda"),
                          t=torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)),
                          grad=torch.empty(n, device="cuda"), aux=torch.zeros(1, device="cuda"))
        a, b, c = mk(), mk(), mk()
        counter = torch.zeros(1, dtype=torch.int32, device="cuda"); status = torch.zeros(1, dtype=torch.int32, device="cuda")
        epoch = 1
        for step in range(1, 5):
            work = torch.randn((parts, n + 1), device="cuda", generator=g) * 1e-2
            args = (step, 1e-3, 0.9, 0.999, 1e-7, 0.25, 1.0)
            check(lib.ss_reduce_adam_tf(work.data_ptr(), parts, n, a["aux"].data_ptr(), a["grad"].data_ptr(), a["p"].data_ptr(),
                                        a["m"].data_ptr(), a["v"].data_ptr(), a["t"].data_ptr(), *args, st), "local")
            check(lib.ss_peer_reduce_push(work.data_ptr(), parts, n, b["aux"].data_ptr(), bases, 1, 0, n, epoch, counter.data_ptr(), st),
                  "push")
            check(lib.ss_peer_adam_tf(own, 1, n, epoch, b["p"].data_ptr(), b["m"].data_ptr(), b["v"].data_ptr(), b["t"].data_ptr(),
                                      b["grad"].data_ptr(), n, *args, status.data_ptr(), st), "adam")
            epoch += 1
            check(lib.ss_peer_reduce_adam_tf(work.data_ptr(), parts, n, c["aux"].data_ptr(), bases, 1, 0, n, epoch, c["p"].data_ptr(),
                                             c["m"].data_ptr(), c["v"].data_ptr(), c["t"].data_ptr(), c["grad"].data_ptr(), *args,
                                             status.data_ptr(), st), "fused")
            epoch += 1
            torch.cuda.synchronize()
            for k in a:
                assert torch.equal(a[k], b[k]), (step, "two kernels", k)
                assert torch.equal(a[k], c[k]), (step, "one kernel", k)
        assert int(status) == 0
    finally:
        lib.ss_peer_free(own)
