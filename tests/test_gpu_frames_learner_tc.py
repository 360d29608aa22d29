"""The learner of the frame-stacked networks on the tensor cores (ss_*_frames_tc, ss_frames_grad_tc.cu) against the
torch-CPU oracle (oracle/learner_oracle.py) and against the exact float32 frames path.  Tolerances as for the 12-input
tensor-core kernels (tests/test_gpu_learner_parity.py): gradients to 2e-2 of their scale -- checked per Keras array, so an
error in the dW1 kernel cannot hide behind W3 -- and 2e-2 absolute on q, y and actions."""
import numpy as np
import pytest
import torch

from oracle import learner_oracle as lo
from tests import philox_ref

_TOL = 2e-2


def _arrays_close(got, want, shapes, rel=_TOL):
    for k, (g, w) in enumerate(zip(lo.split(np.asarray(got), shapes), lo.split(np.asarray(want), shapes))):
        scale = np.abs(w).max() + 1e-12
        err = np.abs(g - w).max() / scale
        assert err <= rel, "array %d (shape %s): %.3g of its scale" % (k, w.shape, err)


class _TC:
    """The C entry points at any frames (1 included: ActorCritic keeps the 12-input kernels there)."""

    def __init__(self, frames, theta, phi, n):
        from skillshot_learning_b200 import _lib
        self.L, self.F, self.n = _lib.lib, frames, n
        self.theta = torch.as_tensor(theta, dtype=torch.float32).cuda()
        self.phi = torch.as_tensor(phi, dtype=torch.float32).cuda()
        self.ws = torch.empty(int(self.L.ss_learner_frames_tc_workspace_bytes(frames, n)), dtype=torch.uint8, device="cuda")
        self.stream = torch.cuda.current_stream().cuda_stream

    def _ws(self):
        return self.ws.data_ptr(), self.ws.numel(), self.stream

    def critic_forward(self, s, a):
        q = torch.empty(self.n, device="cuda")
        up = torch.empty((self.n, 2), device="cuda")
        assert self.L.ss_critic_forward_frames_tc(self.phi.data_ptr(), self.F, s.data_ptr(), a.data_ptr(), q.data_ptr(), up.data_ptr(),
                                                  self.n, *self._ws()) == 0
        return q.cpu().numpy(), up.cpu().numpy()

    def targets(self, r, s2, done, gamma):
        y = torch.empty(self.n, device="cuda")
        assert self.L.ss_ddpg_targets_frames_tc(self.theta.data_ptr(), self.phi.data_ptr(), self.F, r.data_ptr(), s2.data_ptr(),
                                                done.data_ptr(), gamma, y.data_ptr(), self.n, *self._ws()) == 0
        return y.cpu().numpy()

    def critic_grad(self, s, a, y, keep=None, seed=0, counter=0, n_global=0, row_offset=0, slices_only=False):
        g = torch.empty(len(self.phi), device="cuda")
        sse = torch.zeros(1, device="cuda")
        rc = self.L.ss_critic_grad_frames_tc(self.phi.data_ptr(), self.F, s.data_ptr(), a.data_ptr(), y.data_ptr(),
                                             None if keep is None else keep.data_ptr(), 0.2, seed, counter, self.n, n_global, row_offset,
                                             None if slices_only else g.data_ptr(), sse.data_ptr(), *self._ws())
        if slices_only:
            assert rc > 0
            return rc
        assert rc == 0
        return g.cpu().numpy(), float(sse)

    def actor_grad(self, s):
        g = torch.empty(len(self.theta), device="cuda")
        qs = torch.zeros(1, device="cuda")
        assert self.L.ss_actor_grad_frames_tc(self.theta.data_ptr(), self.phi.data_ptr(), self.F, s.data_ptr(), self.n, g.data_ptr(),
                                              qs.data_ptr(), *self._ws()) == 0
        return g.cpu().numpy(), float(qs)


def _setup(frames, n, seed=0):
    rng = np.random.default_rng(seed)
    theta, phi = lo.init_actor(rng, frames), lo.init_critic(rng, frames)
    s = rng.uniform(0, 1, (n, 12 * frames)).astype(np.float32)
    a = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
    y = (-rng.uniform(0, 1, n)).astype(np.float32)
    return rng, theta, phi, s, a, y


@pytest.mark.gpu
@pytest.mark.parametrize("n", [203, 4173])
@pytest.mark.parametrize("frames", [1, 4, 20])
def test_frames_tc_matches_the_oracle(frames, n):
    rng, theta, phi, s, a, y = _setup(frames, n)
    tc = _TC(frames, theta, phi, n)
    S, A, Y = (torch.from_numpy(x).cuda() for x in (s, a, y))
    ashapes, cshapes = lo.actor_shapes(frames), lo.critic_shapes(frames)
    # critic forward: q and -dQ/da
    q, up = tc.critic_forward(S, A)
    np.testing.assert_allclose(q, lo.critic_forward(phi, s, a), rtol=0, atol=_TOL)
    phi_t = torch.tensor(phi, dtype=torch.float64)
    a_t = torch.tensor(a, dtype=torch.float64, requires_grad=True)
    lo.critic_forward_t(phi_t, torch.tensor(s, dtype=torch.float64), a_t).sum().backward()
    # -dQ/da sums W3[k] W2[256 + m][k] in fp32 over the ACTIVE hidden-2 units; only which units are active depends on the
    # bf16 layer 2.  A unit within rounding of zero can flip and move a row by one such term (a few per cent of the rows
    # see one): the worst row is bounded by a few terms, and the mean stays tight.
    want, scale = -a_t.grad.numpy(), np.abs(a_t.grad.numpy()).max()
    _, _, w2, _, w3, _ = lo.split(phi, cshapes)
    term = np.abs(w3[:, 0] * w2[256:258]).max()
    err = np.abs(up - want)
    assert err.max() <= 3 * term + 1e-4
    assert err.mean() <= 1e-2 * scale + 5e-4
    # critic gradient: injected mask, then Philox dropout
    keep = (rng.uniform(size=(n, 256)) >= 0.2).astype(np.uint8)
    g, sse = tc.critic_grad(S, A, Y, keep=torch.from_numpy(keep).cuda())
    want, want_sse = lo.critic_grad(phi, s, a, y, keep.astype(np.float32))
    _arrays_close(g, want, cshapes)
    assert abs(sse - want_sse) <= _TOL * max(1.0, want_sse)
    g, sse = tc.critic_grad(S, A, Y, seed=7, counter=5)
    want, want_sse = lo.critic_grad(phi, s, a, y, philox_ref.dropout_keep(n, 7, 5, 0.2).astype(np.float32))
    _arrays_close(g, want, cshapes)
    assert abs(sse - want_sse) <= _TOL * max(1.0, want_sse)
    # actor gradient and sum q
    g, qs = tc.actor_grad(S)
    want, want_q = lo.actor_grad(theta, phi, s)
    # the actor's upstream gradient is the critic's -dQ/da, whose flipped units (above) move single rows; over 203 rows
    # such a row is not averaged out and dW2 lands at up to ~2.3 % of its scale at 20 frames
    _arrays_close(g, want, ashapes, rel=_TOL if n > 1000 else 3e-2)
    assert abs(qs - want_q) <= _TOL * max(1.0, abs(want_q))
    # TD targets with a done mask, gamma = 0.9
    done = (rng.uniform(size=n) < 0.3).astype(np.uint8)
    yy = tc.targets(Y, S, torch.from_numpy(done).cuda(), 0.9)
    np.testing.assert_allclose(yy, lo.ddpg_targets(theta, phi, y, s, done, 0.9), rtol=0, atol=_TOL)


@pytest.mark.gpu
def test_frames_tc_against_the_float32_path_at_scale():
    """20 frames, 65,536 + 77 rows: many tiles per CTA, every SM, a ragged last tile."""
    from skillshot_learning_b200 import ActorCritic
    F, n = 20, 65536 + 77
    _, theta, phi, s, a, y = _setup(F, n, seed=4)
    nets = [ActorCritic(device="cuda:0", seed=3, frames=F, gamma=0.9, update_precision=p) for p in ("f32", "bf16")]
    out = []
    for ac in nets:
        ac.set_weights(theta, phi)
        gc = ac.critic_grad(s, a, y).cpu().numpy().copy()
        ga = ac.actor_grad(s).cpu().numpy().copy()
        yy = ac.td_targets(y, s).cpu().numpy()
        q = ac.critic_forward(s, a, precision=ac.update_precision).cpu().numpy()
        out.append((gc, ga, yy, q, float(ac.stats[0]), float(ac.stats[1])))
    (gc0, ga0, y0, q0, sse0, qs0), (gc1, ga1, y1, q1, sse1, qs1) = out
    _arrays_close(gc1, gc0, lo.critic_shapes(F))
    _arrays_close(ga1, ga0, lo.actor_shapes(F))
    np.testing.assert_allclose(y1, y0, rtol=0, atol=_TOL)
    np.testing.assert_allclose(q1, q0, rtol=0, atol=_TOL)
    assert abs(sse1 - sse0) <= _TOL * sse0 and abs(qs1 - qs0) <= _TOL * max(1.0, abs(qs0))


@pytest.mark.gpu
def test_frames_tc_slices_determinism_and_sharding():
    from skillshot_learning_b200 import ActorCritic
    F, n = 20, 9000
    _, theta, phi, s, a, y = _setup(F, n, seed=5)
    ac = ActorCritic(device="cuda:0", seed=3, frames=F, update_precision="bf16")
    ac.set_weights(theta, phi)
    S, A, Y = (torch.from_numpy(x).cuda() for x in (s, a, y))
    c0 = ac.counter
    g1 = ac.critic_grad(S, A, Y).clone()
    ac.counter = c0                                          # the same dropout draw again
    g2 = ac.critic_grad(S, A, Y).clone()
    assert torch.equal(g1, g2)                               # fixed-order sums: identical bits
    # slices + the reduce/Adam kernel's gradient output: the same bits as the grad_out path
    ac.counter = c0
    parts = ac.critic_grad(S, A, Y, slices_only=True)
    ac.reduce_adam("critic", parts, None)
    assert torch.equal(ac._slice(ac.grads, "critic"), g1)
    ga = ac.actor_grad(S).clone()
    parts = ac.actor_grad(S, slices_only=True)
    ac.reduce_adam("actor", parts, None)
    assert torch.equal(ac._slice(ac.grads, "actor"), ga)
    # two half batches with n_global / row_offset sum to the full batch (same dropout rows), to fp32 reordering
    ac2 = ActorCritic(device="cuda:0", seed=3, frames=F, update_precision="bf16")
    ac2.set_weights(theta, phi)
    c0 = ac2.counter
    full = ac2.critic_grad(S, A, Y).clone()
    h = 4480                                                  # a multiple of the 128-row tile: the same tiles of bf16 rounding
    parts = []
    for lo_, hi_ in ((0, h), (h, n)):
        ac2.counter = c0                                      # the shards of one batch draw with the batch's counter
        parts.append(ac2.critic_grad(S[lo_:hi_], A[lo_:hi_], Y[lo_:hi_], n_global=n, row_offset=lo_).clone())
    total = (parts[0] + parts[1]).cpu().numpy()
    _arrays_close(total, full.cpu().numpy(), lo.critic_shapes(F), rel=1e-4)


@pytest.mark.gpu
def test_frames_tc_update_tracks_the_float32_update():
    """Twenty updates of 20-frame networks with the tensor-core kernels against the float32 kernels on the same
    minibatches and masks: the losses and q track within the 12-input tensor-core test's tolerance."""
    from skillshot_learning_b200 import ActorCritic
    F, n = 20, 4096
    rng, theta, phi, _, _, _ = _setup(F, 8)
    nets = [ActorCritic(device="cuda:0", seed=1, frames=F, gamma=0.9, tau=0.05, update_precision=p) for p in ("f32", "bf16")]
    for ac in nets:
        ac.set_weights(theta, phi)
    losses, qs = [[], []], [[], []]
    for it in range(20):
        s = torch.from_numpy(rng.uniform(0, 1, (n, 12 * F)).astype(np.float32)).cuda()
        s2 = torch.from_numpy(rng.uniform(0, 1, (n, 12 * F)).astype(np.float32)).cuda()
        a = torch.from_numpy(rng.uniform(-1, 1, (n, 2)).astype(np.float32)).cuda()
        r = torch.from_numpy((-rng.uniform(0, 1, n)).astype(np.float32)).cuda()
        keep = torch.from_numpy((rng.uniform(size=(n, 256)) >= 0.2).astype(np.uint8)).cuda()
        for k, ac in enumerate(nets):
            y = ac.td_targets(r, s2)
            losses[k].append(float(ac.critic_step(s, a, y, keep=keep)) / n)
            qs[k].append(float(ac.actor_step(s)) / n)
    np.testing.assert_allclose(losses[1], losses[0], rtol=3e-2, atol=1e-4)
    np.testing.assert_allclose(qs[1], qs[0], rtol=3e-2, atol=1e-4)


@pytest.mark.gpu
def test_frames_tc_selfplay_trainer():
    from skillshot_learning_b200 import SelfPlayTrainer
    F, n = 4, 256
    kw = dict(device="cuda:0", seed=11, frames=F, batch_size=512, replay_capacity=2 * n * 8, noise_group=128, tick_limit=9,
              gamma=0.9, tau=0.05, precision="bf16", param_noise_sd=0.5)
    assert SelfPlayTrainer(n, **kw).networks.update_precision == "f32"          # the default mapping is unchanged
    tr = SelfPlayTrainer(n, update_precision="bf16", **kw)
    assert tr.networks.update_precision == "bf16"
    tr.rollout(5)
    net = tr.networks
    theta, phi = net.target_actor.cpu().numpy().copy(), net.target_critic.cpu().numpy().copy()
    phi_online = net.critic.cpu().numpy().copy()
    counter = net.counter
    tr.update()
    b = tr._batch
    bs, ba, br, bn, bd = (b[k].cpu().numpy() for k in ("obs", "act", "reward", "next_obs", "done"))
    y = lo.ddpg_targets(theta, phi, br, bn, bd, 0.9)
    keep = philox_ref.dropout_keep(512, net.seed, counter, 0.2)
    gq, _ = lo.critic_grad(phi_online, bs, ba, y, keep.astype(np.float32))
    _arrays_close(net.grads[net._c_off:net._c_off + net.c_n].cpu().numpy(), gq, lo.critic_shapes(F))
    assert torch.isfinite(net.params).all()
    # checkpoint round trip: the resumed trainer updates bit-identically
    sd = tr.state_dict()
    assert sd["update_precision"] == "bf16"
    tr2 = SelfPlayTrainer(n, update_precision="bf16", **kw)
    tr2.load_state_dict(sd)
    for t in (tr, tr2):
        t.rollout(2)
        t.update()
    assert torch.equal(tr.networks.params, tr2.networks.params)
    old = {k: v for k, v in sd.items() if k != "update_precision"}          # a checkpoint written before the field existed
    tr3 = SelfPlayTrainer(n, **kw)
    tr3.load_state_dict(old)
    assert tr3.update_precision is None


def test_frames_tc_entry_points_reject_invalid_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L = _lib.lib
    need = L.ss_learner_frames_tc_workspace_bytes(20, 65536)
    tiles, pn = 512, 240 * 256 + 256 + 258 * 128 + 128 + 128 + 1            # the critic is the larger network
    x, h = tiles * 32 * 2048, tiles * 65536
    assert need == (tiles * (pn + 1) * 4 + 15) // 16 * 16 + 3 * x + 2 * h + 65536 * 8 * 2 + 65536 * 4
    assert L.ss_learner_frames_tc_workspace_bytes(0, 16) == -1 and L.ss_learner_frames_tc_workspace_bytes(21, 16) == -1
    assert L.ss_learner_frames_tc_workspace_bytes(4, 0) == -1
    p, ws = 4096, 1 << 30                                     # aligned fake addresses: rejected before any device call
    assert L.ss_critic_forward_frames_tc(None, 4, p, p, p, None, 16, p, ws, None) == -1
    assert L.ss_critic_forward_frames_tc(p, 21, p, p, p, None, 16, p, ws, None) == -1
    assert L.ss_critic_forward_frames_tc(p, 4, p, p, p, None, 16, p + 8, ws, None) == -1          # misaligned workspace
    assert L.ss_critic_forward_frames_tc(p, 4, p, p, p, None, 16, p, 1024, None) == -1            # short workspace
    assert L.ss_ddpg_targets_frames_tc(p, p, 0, p, p, None, 0.9, p, 16, p, ws, None) == -1
    assert L.ss_ddpg_targets_frames_tc(p, p, 4, None, p, None, 0.9, p, 16, p, ws, None) == -1
    assert L.ss_critic_grad_frames_tc(p, 4, p, p, p, None, 1.0, 0, 0, 16, 16, 0, None, None, p, ws, None) == -1
    assert L.ss_critic_grad_frames_tc(p, 4, p + 4, p, p, None, 0.2, 0, 0, 16, 16, 0, None, None, p, ws, None) == -1
    assert L.ss_critic_grad_frames_tc(p, 4, p, p, p, None, 0.2, 0, 0, 0, 16, 0, None, None, p, ws, None) == -1
    assert L.ss_actor_grad_frames_tc(p, None, 4, p, 16, None, None, p, ws, None) == -1
    assert L.ss_actor_grad_frames_tc(p, p, 4, p, 16, None, None, None, ws, None) == -1
    assert L.ss_actor_grad_frames_tc(p, p, 4, p, 16, None, None, p, L.ss_learner_frames_tc_workspace_bytes(4, 16) - 1, None) == -1
