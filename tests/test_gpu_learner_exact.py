"""The tensor-core learner kernels (ss_*_tc, ss_*_frames_tc) and their float32 counterparts against float64 autograd
(oracle/learner_oracle.py, tests/td3_oracle.py) on networks and batches on which every rounding the kernels do is exact
(tests/exact_nets.py; tests/test_exact_nets.py checks that premise at every shape used here).  A correct kernel returns the
float64 answer, so every comparison is ==; the one exception is the actor's output, which goes through tanhf and is compared
within its 2-ulp bound (everything before tanh is exact).  A difference while the premise holds is a kernel bug."""
import numpy as np
import pytest
import torch

from oracle import learner_oracle as lo
from tests import exact_nets as xn
from tests.td3_oracle import td3_targets

pytestmark = pytest.mark.gpu
F64 = torch.float64


def _cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _same(got, want, what, shapes=None):
    """got == want elementwise; on a difference name the first differing value (and its Keras array)."""
    got, want = np.asarray(got, np.float64).ravel(), np.asarray(want, np.float64).ravel()
    assert got.shape == want.shape, what
    bad = np.flatnonzero(got != want)
    if bad.size == 0:
        return
    where = ""
    if shapes is not None:
        ends = np.cumsum([int(np.prod(s)) for s in shapes])
        k = int(np.searchsorted(ends, bad[0], side="right"))
        where = " (array %d, shape %s)" % (k, shapes[k])
    raise AssertionError("%s: %d of %d values differ; first at %d%s: %r, want %r" % (
        what, bad.size, got.size, bad[0], where, got[bad[0]], want[bad[0]]))


def _tanh_close(got, want, what):
    """Within 2 float32 ulp of float64 tanh: the documented bound of tanhf."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    err = np.abs(got - want) / ulp
    assert err.max() <= 2.0, "%s: %.2f ulp" % (what, err.max())


class _Entry:
    """The C entry points on one batch of tests/exact_nets.py.  frames_api: the frame-stacked entry points (any frames,
    1 included); else the 12-input ones (frames = 1).  tc: tensor cores, else the float32 kernels."""

    def __init__(self, b, tc, frames_api):
        from skillshot_learning_b200 import _lib
        self.L, self.F, self.n = _lib.lib, b["frames"], b["n"]
        self.tc, self.fr = tc, frames_api
        assert frames_api or self.F == 1
        self.st = torch.cuda.current_stream().cuda_stream
        L, F, n = self.L, self.F, self.n
        pn = max(L.ss_actor_frames_params(F), L.ss_critic_frames_params(F))
        ws = max(L.ss_learner_workspace_bytes() + 32 * n, L.ss_learner_frames_tc_workspace_bytes(F, n), 160 * (pn + 1) * 4)
        self.ws = torch.empty(ws, dtype=torch.uint8, device="cuda")

    def _ws(self):
        return self.ws.data_ptr(), self.ws.numel()

    def critic_forward(self, phi, s, a):
        L, n = self.L, self.n
        q = torch.empty(n, device="cuda")
        up = torch.empty((n, 2), device="cuda") if self.tc else None
        P, S, A = (t.data_ptr() for t in (phi, s, a))
        if self.tc and self.fr:
            rc = L.ss_critic_forward_frames_tc(P, self.F, S, A, q.data_ptr(), up.data_ptr(), n, *self._ws(), self.st)
        elif self.tc:
            rc = L.ss_critic_forward_tc(P, S, A, n, q.data_ptr(), up.data_ptr(), None, None, 0.0, None, self.st)
        elif self.fr:
            rc = L.ss_critic_forward_frames(P, self.F, S, A, q.data_ptr(), n, self.st)
        else:
            rc = L.ss_critic_forward(P, S, A, q.data_ptr(), n, self.st)
        assert rc == 0
        return q.cpu().numpy(), None if up is None else up.cpu().numpy()

    def ddpg_targets(self, theta, phi, r, s2, done):
        L, n = self.L, self.n
        y = torch.empty(n, device="cuda")
        T, P, R, S2, D = (t.data_ptr() for t in (theta, phi, r, s2, done))
        if self.tc and self.fr:
            rc = L.ss_ddpg_targets_frames_tc(T, P, self.F, R, S2, D, xn.GAMMA, y.data_ptr(), n, *self._ws(), self.st)
        elif self.tc:
            rc = L.ss_ddpg_targets_tc(T, P, R, S2, D, xn.GAMMA, y.data_ptr(), n, *self._ws(), self.st)
        elif self.fr:
            rc = L.ss_ddpg_targets_frames(T, P, self.F, R, S2, D, xn.GAMMA, y.data_ptr(), n, self.st)
        else:
            rc = L.ss_ddpg_targets(T, P, R, S2, D, xn.GAMMA, y.data_ptr(), n, self.st)
        assert rc == 0
        return y.cpu().numpy()

    def td3_targets(self, theta, phi, phi2, r, s2, done):
        """Two critics, no smoothing noise: y = r + gamma (1 - done) min(q1, q2)."""
        L, n = self.L, self.n
        y = torch.empty(n, device="cuda")
        head = tuple(t.data_ptr() for t in (theta, phi, phi2))
        tail = tuple(t.data_ptr() for t in (r, s2, done)) + (xn.GAMMA, 0.0, 0.5, xn.SEED, 0, 0, y.data_ptr(), n)
        if self.tc and self.fr:
            rc = L.ss_td3_targets_frames_tc(*head, self.F, *tail, *self._ws(), self.st)
        elif self.tc:
            rc = L.ss_td3_targets_tc(*head, *tail, *self._ws(), self.st)
        else:
            rc = L.ss_td3_targets_frames(*head, self.F, *tail, None, 0, self.st)
        assert rc == 0
        return y.cpu().numpy()

    def critic_grad(self, phi, s, a, y, keep=None, n=None, n_global=0, row_offset=0):
        """keep None: the Philox mask of (xn.SEED, xn.COUNTER) keyed by global row row_offset + i."""
        L, n = self.L, self.n if n is None else n
        g = torch.empty(phi.numel(), device="cuda")
        sse = torch.zeros(1, device="cuda")
        args = (tuple(t.data_ptr() for t in (s, a, y)) +
                (None if keep is None else keep.data_ptr(), xn.RATE, xn.SEED, xn.COUNTER, n, n_global, row_offset,
                 g.data_ptr(), sse.data_ptr(), *self._ws(), self.st))
        if self.fr:
            fn = L.ss_critic_grad_frames_tc if self.tc else L.ss_critic_grad_frames
            rc = fn(phi.data_ptr(), self.F, *args)
        else:
            rc = (L.ss_critic_grad_tc if self.tc else L.ss_critic_grad)(phi.data_ptr(), *args)
        assert rc == 0
        return g.cpu().numpy(), float(sse)

    def actor_grad(self, theta, phi, s):
        L, n = self.L, self.n
        g = torch.empty(theta.numel(), device="cuda")
        qs = torch.zeros(1, device="cuda")
        tail = (s.data_ptr(), n, g.data_ptr(), qs.data_ptr(), *self._ws(), self.st)
        if self.fr:
            rc = (L.ss_actor_grad_frames_tc if self.tc else L.ss_actor_grad_frames)(theta.data_ptr(), phi.data_ptr(), self.F, *tail)
        else:
            rc = (L.ss_actor_grad_tc if self.tc else L.ss_actor_grad)(theta.data_ptr(), phi.data_ptr(), *tail)
        assert rc == 0
        return g.cpu().numpy(), float(qs)


def _dq_da(phi, s, a):
    """-dQ/da of every row, float64 autograd."""
    at = torch.tensor(a, dtype=F64, requires_grad=True)
    lo.critic_forward_t(torch.tensor(phi, dtype=F64), torch.tensor(s, dtype=F64), at).sum().backward()
    return -at.grad.numpy()


def _check_learner(b, ent, what):
    """Every learner entry point of `ent` on batch b against float64: critic forward (q, -dQ/da on the tensor cores),
    critic gradient and sum of squared errors under the injected and the Philox mask, policy gradient and sum q, the
    DDPG and the TD3 (two critics) targets."""
    F, n = b["frames"], b["n"]
    d = {k: _cuda(b[k]) for k in ("theta", "phi", "phi_pi", "phi2", "s", "s2", "a", "r", "done")}
    cshapes, ashapes = lo.critic_shapes(F), lo.actor_shapes(F)
    q, up = ent.critic_forward(d["phi"], d["s"], d["a"])
    _same(q, lo.critic_forward(b["phi"], b["s"], b["a"], None, dtype=F64), what + " q")
    if up is not None:
        _same(up, _dq_da(b["phi"], b["s"], b["a"]), what + " -dQ/da")
    ng = xn.n_global(n)
    for name, keep in (("injected", b["keep"]), ("philox", xn.philox_keep(n))):
        y = xn.targets(b, keep)
        g, sse = ent.critic_grad(d["phi"], d["s"], d["a"], _cuda(y), _cuda(keep) if name == "injected" else None, n_global=ng)
        want, want_sse = lo.critic_grad(b["phi"], b["s"], b["a"], y, keep, xn.RATE, ng, dtype=F64)
        _same(g, want, "%s critic gradient, %s mask" % (what, name), cshapes)
        _same(sse, want_sse, "%s sum of squared errors, %s mask" % (what, name))
    g, qs = ent.actor_grad(d["theta"], d["phi_pi"], d["s"])
    want, want_q = lo.actor_grad(b["theta"], b["phi_pi"], b["s"], dtype=F64)
    assert all(np.abs(w).max() > 0 for w in lo.split(want, ashapes))          # the paired actor's backward pass does not cancel
    _same(g, want, what + " policy gradient", ashapes)
    _same(qs, want_q, what + " sum q")
    y = ent.ddpg_targets(d["theta"], d["phi"], d["r"], d["s2"], d["done"])
    _same(y, lo.ddpg_targets(b["theta"], b["phi"], b["r"], b["s2"], b["done"], xn.GAMMA, dtype=F64), what + " DDPG targets")
    if ent.tc and ent.fr and F == 1:
        return                                                                  # ss_td3_targets_frames_tc: frames 2..20
    y = ent.td3_targets(d["theta"], d["phi"], d["phi2"], d["r"], d["s2"], d["done"])
    want = td3_targets(b["theta"], b["phi"], b["phi2"], b["r"], b["s2"], b["done"], xn.GAMMA, dtype=F64)
    _same(y, want, what + " TD3 targets")


@pytest.mark.parametrize("n", xn.ROWS_12)
def test_12_input_learner_kernels_equal_float64(n):
    from skillshot_learning_b200 import _lib
    b = xn.make(1, n)
    # actor forward (unpaired actor): tanhf of an exact pre-activation
    out = torch.empty((n, 2), device="cuda")
    assert _lib.lib.ss_actor_forward_tc(_cuda(b["theta_fwd"]).data_ptr(), _cuda(b["s"]).data_ptr(), out.data_ptr(), n, 0.0, 1, 0.0,
                                        0, 0, torch.cuda.current_stream().cuda_stream) == 0
    _tanh_close(out.cpu().numpy(), lo.actor_forward(b["theta_fwd"], b["s"], dtype=F64), "ss_actor_forward_tc")
    _check_learner(b, _Entry(b, tc=True, frames_api=False), "12-input tensor cores")
    _check_learner(b, _Entry(b, tc=False, frames_api=False), "12-input float32")


@pytest.mark.parametrize("frames,n", [(f, n) for f in range(1, 21) for n in xn.ROWS_FRAMES] +
                         [(f, xn.ROWS_LARGE) for f in xn.FRAMES_LARGE])
def test_frame_stacked_learner_kernels_equal_float64(frames, n):
    """(1, 65,613) is also the layer-1 kernel with one K stage (frames <= 5) and several tiles per CTA: its MMA warp once
    waited for the next tile's operands before releasing the stage they load into, and the launch never finished."""
    from skillshot_learning_b200 import FrameStackActor
    b = xn.make(frames, n)
    # the acting forward reads the fp16 history ring: push the frames oldest first
    fsa = FrameStackActor(n, frames=frames, device="cuda:0", precision="bf16", params=_cuda(b["theta_fwd"]))
    for f in range(frames):
        fsa.push(_cuda(b["s"][:, 12 * f:12 * f + 12]))
    _tanh_close(fsa.forward().cpu().numpy(), lo.frames_actor_forward(b["theta_fwd"], b["s"], frames, dtype=F64),
                "ss_actor_forward_frames_tc")
    _check_learner(b, _Entry(b, tc=True, frames_api=True), "%d-frame tensor cores" % frames)
    _check_learner(b, _Entry(b, tc=False, frames_api=True), "%d-frame float32" % frames)


@pytest.mark.parametrize("frames,n,split", xn.SHARDS)
@pytest.mark.parametrize("tc", [True, False])
def test_shards_of_a_batch_sum_exactly_to_the_batch(frames, n, split, tc):
    """Two shards split inside a 128-row tile, Philox dropout keyed by the global row: each shard's gradient is the float64
    gradient of its rows under the batch's mask, and the two add up to the whole batch's gradient bit for bit."""
    b = xn.make(frames, n)
    ent = _Entry(b, tc=tc, frames_api=frames > 1)
    keep = xn.philox_keep(n)
    y = xn.targets(b, keep)
    ng = xn.n_global(n)
    phi, s, a, yy = _cuda(b["phi"]), _cuda(b["s"]), _cuda(b["a"]), _cuda(y)
    full, _ = ent.critic_grad(phi, s, a, yy, n_global=ng)
    parts = []
    for lo_, hi_ in ((0, split), (split, n)):
        g, _ = ent.critic_grad(phi, s[lo_:hi_], a[lo_:hi_], yy[lo_:hi_], n=hi_ - lo_, n_global=ng, row_offset=lo_)
        want, _ = lo.critic_grad(b["phi"], b["s"][lo_:hi_], b["a"][lo_:hi_], y[lo_:hi_], keep[lo_:hi_], xn.RATE, ng, dtype=F64)
        _same(g, want, "shard %d..%d" % (lo_, hi_), lo.critic_shapes(frames))
        parts.append(g)
    _same(parts[0] + parts[1], full, "the two shards' sum", lo.critic_shapes(frames))
