"""Networks and batches on which every rounding of the tensor-core learner kernels is exact.

The tensor-core kernels (ss_mlp_tc.cu, ss_mlp_grad_tc.cu, ss_frames_tc.cu, ss_frames_grad_tc.cu) round their GEMM operands
to fp16 (forward layer 1) or bf16 (everything else; observations, actions, biases and the output-layer gradient as hi + lo
pairs) and accumulate in fp32.  On the inputs built here each of those roundings is the identity and each fp32 sum is exact in
any order, so a correct kernel returns the float64 answer of oracle/learner_oracle.py bit for bit, whatever its tiling,
summation order or slice count.  No model of the kernels' rounding is involved: check_* recompute every intermediate in
float64 and assert the premise, which tests/test_exact_nets.py does at every shape tests/test_gpu_learner_exact.py uses.

The premise, per operand and per sum:
  * an fp16 operand has at most 11 significant bits, a bf16 operand at most 8, a hi + lo pair at most 16;
  * the terms of an fp32 sum are multiples of one grid unit u and their absolute values add up to less than 2^24 u;
  * dropout rate 0.5 (scale 2), gamma 0.5, n_global a power of two: every scalar factor is a power of two;
  * no ReLU pre-activation is exactly zero (biases on half-grid offsets), so the derivative convention at 0 never matters.

Construction:
  * observations in {0, 1}; two "fine" columns carry 1 + k 2^-9 (k = 1, 2) on sparse rows (and the last row).  Their bf16
    high half is 1, so the signal is in the low half.  Each fine column feeds one hidden-1 unit alone, with weight 512 and
    bias -511.5: its pre-activation is k + 0.5, i.e. carried by the observation's low half, and the bias' own bf16 low half
    (0.5) matters too.  The fine columns stay zero elsewhere so that their weight-gradient sums keep within 24 bits.
  * the critic's first action column is 0 except on the sparse rows, where it is 0.5 + k 2^-10 (high half 0.5), -0.5 or -1;
    it feeds one hidden-2 unit alone, weight 1024 and bias -511.5.  The second action column is in {+-0.5, +-1}.
  * W1 in {-1, 0, 1} with about 12 % / sqrt(frames) non-zero; W2 in {-2, 0, 2} (even, so that half-integer activations give
    integer sums); critic W3 = +-1; biases in Z + 1/2; targets y = q - e with e in {+-1, +-2} on every row.
  * the actor of the gradient and target tests returns exactly 0: hidden-1 units come in pairs with identical W1 columns and
    biases, hidden-2 units in pairs (u, u') with W2[:, u'] = W2[:, u] + beta (e_p - e_p') for one hidden-1 pair (p, p'),
    W3[u'] = -W3[u] and b3 = 0.  Then z3 = 0 and tanhf(0) = 0 exactly, while the backward pass does not cancel:
    dz1[p] = -dz1[p'] != 0, so every actor gradient array is non-zero.  Its critic (phi_pi) has a dense first action row,
    which the critic tests' critic cannot have: at a = 0 no low half is involved.  On small batches phi_pi also gives the
    actor's upstream gradient values of 9 bits, so that dz3 needs its low half (policy_critic).
  * the actor of the forward tests is unpaired, W3 = +-2^-6 (sparse), so tanh sees values of order 1; its output is compared
    within tanhf's error bound, everything before tanh exactly.
"""
import numpy as np

from oracle import learner_oracle as lo

H1, H2 = 256, 128
RATE, GAMMA = 0.5, 0.5
SEED, COUNTER = 11, 5                  # Philox key of the dropout masks
FINE_EVERY, FINE_PHASE = 509, 5        # rows r % 509 == 5, and the last row, carry the low-half inputs
FINE_UP_ROWS = 1024                    # batches up to this size also give the actor's dz3 a low half (policy_critic)

# the shapes of tests/test_gpu_learner_exact.py: tile edges, one row either side of a wave of 148 tiles, CTAs of 2-4 rounds
ROWS_12 = (1, 77, 127, 128, 129, 4173, 148 * 128 - 1, 148 * 128 + 1, 3 * 148 * 128 + 77, 65536 + 77)
ROWS_FRAMES = (203, 4173)              # at every frame count 1..20: every K1 = round16(12 F + 2) from 16 to 256
FRAMES_LARGE, ROWS_LARGE = (1, 11, 20), 65536 + 77
SHARDS = ((1, 4173, 1701), (20, 4173, 1701))      # (frames, rows, split row): a split inside a 128-row tile


def n_global(n):
    """The loss divisor: the next power of two >= n, so that 2 e / n_global is exact."""
    return 1 << (int(n) - 1).bit_length()


def fine_rows(n):
    return np.unique(np.r_[np.arange(FINE_PHASE, n, FINE_EVERY), n - 1])


def fine_cols(frames):
    return [10, 12 * frames - 1]       # column 10 of the oldest frame, column 11 of the newest


# ---------------------------------------------------------------------------------------------------------------------
# parameters
# ---------------------------------------------------------------------------------------------------------------------
def _layer1(rng, frames, paired):
    k = 12 * frames
    fc = fine_cols(frames)
    coarse = [c for c in range(k) if c not in fc]
    w1 = np.zeros((k, H1))
    w1[coarse] = rng.choice([-1.0, 1.0], (len(coarse), H1)) * (rng.uniform(size=(len(coarse), H1)) < 0.12 / np.sqrt(frames))
    b1 = rng.choice([-1.5, -0.5, 0.5, 1.5], H1)
    for i, c in enumerate(fc):         # units 0 and 2: the fine columns' own units
        p = 2 * i
        w1[:, p] = 0.0
        w1[c, p] = 512.0
        b1[p] = -511.5
    if paired:
        w1[:, 1::2] = w1[:, 0::2]
        b1[1::2] = b1[0::2]
    return w1, b1


def _w2(rng, rows, density=0.04):
    return rng.choice([-2.0, 2.0], (rows, H2)) * (rng.uniform(size=(rows, H2)) < density)


def _b2(rng):
    return rng.choice([-2.5, -1.5, -0.5, 0.5, 1.5, 2.5], H2)


def _flat(parts):
    return np.concatenate([np.asarray(p, np.float64).ravel() for p in parts]).astype(np.float32)


def critic_params(rng, frames):
    """The critic of the critic tests: hidden-2 unit 0 reads the first action column alone (weight 1024, bias -511.5)."""
    w1, b1 = _layer1(rng, frames, paired=False)
    w2 = np.zeros((H1 + 2, H2))
    w2[:H1] = _w2(rng, H1)
    w2[H1 + 1] = rng.choice([-2.0, 2.0], H2) * (rng.uniform(size=H2) < 0.25)
    b2 = _b2(rng)
    w2[:, 0] = 0.0
    w2[H1, 0], b2[0] = 1024.0, -511.5
    w3 = rng.choice([-1.0, 1.0], (H2, 1))
    return _flat([w1, b1, w2, b2, w3, [0.5]])


def policy_critic(phi, rng, frames, n):
    """phi with a dense first action row {-2, 0, 2}: the critic of the policy-gradient tests, where a = 0.  Up to
    FINE_UP_ROWS rows, hidden-2 units 1 and 3 read no hidden-1 unit, are active on every row and add -(256 + 1) to the
    actor's upstream gradient on its first output and +(256 + 1) on its second: the first has more than bf16's 8 bits
    (dz3 needs its low half) while their sum, which dz2 sees through W3 rows (w, w), stays small.  On more rows the
    dW3 sums of those 9-bit values would need more than fp32's 24 bits."""
    w1, b1, w2, b2, w3, b3 = [x.copy() for x in lo.split(phi.astype(np.float64), lo.critic_shapes(frames))]
    w2[H1] = rng.choice([-2.0, 2.0], H2) * (rng.uniform(size=H2) < 0.25)
    if n <= FINE_UP_ROWS:
        for u, c in ((1, 256.0), (3, 1.0)):
            w2[:, u] = 0.0
            w2[H1, u], w2[H1 + 1, u], b2[u], w3[u] = c, -c, 0.5, 1.0
    return _flat([w1, b1, w2, b2, w3, b3])


def paired_actor(rng, frames):
    """An actor whose output is exactly 0 on every input, with a backward pass that does not cancel (module docstring)."""
    w1, b1 = _layer1(rng, frames, paired=True)
    w2 = np.zeros((H1, H2))
    w2[:, 0::2] = _w2(rng, H1, 0.04)[:, :H2 // 2]
    w2[:, 1::2] = w2[:, 0::2]
    for j in range(H2 // 2):
        p = 2 * int(rng.integers(H1 // 2))
        beta = rng.choice([-2.0, 2.0])
        w2[p, 2 * j + 1] += beta
        w2[p + 1, 2 * j + 1] -= beta
    b2 = _b2(rng)
    b2[1::2] = b2[0::2]
    w3 = np.zeros((H2, 2))
    w3[0::2] = rng.choice([-1.0, 1.0], (H2 // 2, 1))          # rows (w, w): dz2 = w (up0 + up1)
    w3[1::2] = -w3[0::2]
    return _flat([w1, b1, w2, b2, w3, [0.0, 0.0]])


def forward_actor(rng, frames):
    """An unpaired actor for the forward tests: tanh sees values of order 1."""
    w1, b1 = _layer1(rng, frames, paired=False)
    w3 = rng.choice([-1.0, 1.0], (H2, 2)) * 2.0 ** -6 * (rng.uniform(size=(H2, 2)) < 0.25)
    return _flat([w1, b1, _w2(rng, H1), _b2(rng), w3, rng.choice([-1.0, 1.0], 2) * 2.0 ** -4])


# ---------------------------------------------------------------------------------------------------------------------
# batches
# ---------------------------------------------------------------------------------------------------------------------
def observations(rng, n, frames):
    s = (rng.uniform(size=(n, 12 * frames)) < 0.5).astype(np.float64)
    fc, fr = fine_cols(frames), fine_rows(n)
    s[:, fc] = 0.0
    s[np.ix_(fr, fc)] = rng.choice([0.0, 1.0 + 2.0 ** -9, 1.0 + 2.0 ** -8], (len(fr), len(fc)))
    return s.astype(np.float32)


def actions(rng, n):
    a = np.zeros((n, 2))
    a[:, 1] = rng.choice([-1.0, -0.5, 0.5, 1.0], n)
    fr = fine_rows(n)
    a[fr, 0] = rng.choice([0.5 + 2.0 ** -10, 0.5 + 2.0 ** -9, -0.5, -1.0], len(fr))
    return a.astype(np.float32)


def make(frames, n, seed=0):
    """Networks and a batch of n rows for `frames`-frame networks (frames = 1: the 12-input ones).
    keep: an injected dropout mask; e: the per-row error the critic targets are built with (targets())."""
    rng = np.random.default_rng(1000 * frames + seed)
    phi = critic_params(rng, frames)
    return dict(
        frames=frames, n=n,
        theta=paired_actor(rng, frames), theta_fwd=forward_actor(rng, frames),
        phi=phi, phi_pi=policy_critic(phi, rng, frames, n), phi2=critic_params(rng, frames),
        s=observations(rng, n, frames), s2=observations(rng, n, frames), a=actions(rng, n),
        r=rng.choice([-1.0, -0.5, 0.0, 0.25], n).astype(np.float32),
        done=(rng.uniform(size=n) < 0.3).astype(np.uint8),
        keep=(rng.uniform(size=(n, H1)) < 0.5).astype(np.uint8),
        e=rng.choice([-2.0, -1.0, 1.0, 2.0], n))


def targets(b, keep):
    """y = q - e with q the critic's training-mode output under `keep`: every row's error is e."""
    import torch
    q = lo.critic_forward(b["phi"], b["s"], b["a"], keep, RATE, dtype=torch.float64)
    return (q - b["e"]).astype(np.float32)


def philox_keep(n, row_offset=0):
    from tests import philox_ref
    return philox_ref.dropout_keep(n, SEED, COUNTER, RATE, row_offset)


# ---------------------------------------------------------------------------------------------------------------------
# the premise, checked in float64
# ---------------------------------------------------------------------------------------------------------------------
def _need(ok, what):
    if not np.all(ok):
        raise AssertionError("not exact: " + what)


def _lsb(x):
    """Value of the lowest set bit of every element of a float32-exact array (inf for 0)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    ex = (u >> np.uint32(23)) & np.uint32(0xFF)
    m = (u & np.uint32(0x7FFFFF)) | np.where(ex > 0, np.uint32(0x800000), np.uint32(0))
    low = m & (~m + np.uint32(1))
    return np.where(m == 0, np.inf, np.ldexp(low.astype(np.float32), np.maximum(ex.astype(np.int32), 1) - 150).astype(np.float64))


def _bf16(x):
    """Round to nearest even bfloat16 (x already float32-exact)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    u = (u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)
    return u.view(np.float32).astype(np.float64).reshape(np.shape(x))


def _f32(x, what):
    x = np.asarray(x, np.float64)
    _need(x.astype(np.float32).astype(np.float64) == x, what + " in float32")
    return x


def _bf16_exact(x, what):
    x = _f32(x, what)
    _need(_bf16(x) == x, what + " in bf16")


def _bf16_pair(x, what):
    x = _f32(x, what)
    lo_ = x - _bf16(x)
    _need(_bf16(lo_) == lo_, what + " as a bf16 hi + lo pair")


def _f16_exact(x, what):
    x = _f32(x, what)
    _need(x.astype(np.float16).astype(np.float64) == x, what + " in fp16")


def _f16_pair(x, what):
    x = _f32(x, what)
    lo_ = x - x.astype(np.float16).astype(np.float64)
    _need(lo_.astype(np.float16).astype(np.float64) == lo_, what + " as an fp16 hi + lo pair")


def _sum_exact(a, b, bias=None, what=""):
    """a @ b (+ bias) is exact in fp32 in any order: per output, the terms share the grid lsb(row of a) * lsb(column of b)
    (and lsb(bias)), and their absolute values add up to less than 2^24 of it."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    grid = _lsb(a).min(axis=1)[:, None] * _lsb(b).min(axis=0)[None, :]
    bound = np.abs(a) @ np.abs(b)
    if bias is not None:
        bias = np.asarray(bias, np.float64).reshape(1, -1)
        grid = np.minimum(grid, _lsb(bias))
        bound = bound + np.abs(bias)
    _need(bound < 2.0 ** 24 * grid, what + ": fp32 sum")
    return a @ b + (0.0 if bias is None else bias)


def _rows_exact(x, d, what):
    """sum over the rows of x[r, i] d[r, j] (weight gradients, bias gradients with x = 1) is exact."""
    return _sum_exact(np.asarray(x, np.float64).T, d, what=what)


def _layer1_exact(s, w1, b1, what):
    _f16_exact(s, what + " observations")
    _bf16_pair(s, what + " observations")
    _f16_exact(w1, what + " W1")
    _bf16_exact(w1, what + " W1")
    _f16_pair(b1, what + " b1")
    _bf16_pair(b1, what + " b1")
    z1 = _sum_exact(s, w1, b1, what + " z1")
    _need(z1 != 0, what + ": a layer-1 pre-activation is 0")
    h1 = np.maximum(z1, 0.0)
    _bf16_exact(h1, what + " h1")
    return h1


def critic_forward(phi, s, a, keep, frames):
    """The critic's intermediates (keep None: Dropout off), asserting the premise on the way."""
    w1, b1, w2, b2, w3, b3 = lo.split(np.asarray(phi, np.float64), lo.critic_shapes(frames))
    h1 = _layer1_exact(s, w1, b1, "critic")
    x2 = h1 if keep is None else h1 * keep * (1.0 / (1.0 - RATE))
    _bf16_exact(x2, "critic h1 after dropout")
    _bf16_exact(w2, "critic W2")
    _bf16_pair(a, "actions")
    _bf16_pair(b2, "critic b2")
    xa = np.concatenate([x2, np.asarray(a, np.float64)], axis=1)
    z2 = _sum_exact(xa, w2, b2, "critic z2")
    _need(z2 != 0, "critic: a layer-2 pre-activation is 0")
    h2 = np.maximum(z2, 0.0)
    _bf16_exact(h2, "critic h2")
    q = _sum_exact(h2, w3, b3, "critic q")[:, 0]
    wa = w3[:, 0][:, None] * w2[H1:].T                         # [H2, 2]: W3[k] W2[256 + m][k]
    _f32(wa, "W3 W2[action]")
    up = -_sum_exact((z2 > 0).astype(np.float64), wa, what="-dQ/da")
    return dict(x2=x2, xa=xa, z2=z2, h2=h2, q=q, up=up, w2=w2, w3=w3)


def actor_forward(theta, s, frames, paired):
    w1, b1, w2, b2, w3, b3 = lo.split(np.asarray(theta, np.float64), lo.actor_shapes(frames))
    h1 = _layer1_exact(s, w1, b1, "actor")
    _bf16_exact(w2, "actor W2")
    _bf16_pair(b2, "actor b2")
    z2 = _sum_exact(h1, w2, b2, "actor z2")
    _need(z2 != 0, "actor: a layer-2 pre-activation is 0")
    h2 = np.maximum(z2, 0.0)
    _bf16_exact(h2, "actor h2")
    z3 = _sum_exact(h2, w3, b3, "actor z3")
    if paired:
        _need(z3 == 0, "the paired actor's output layer is not 0")
    return dict(h1=h1, z2=z2, h2=h2, z3=z3, w2=w2, w3=w3)


def check_critic_grad(phi, s, a, y, keep, ng, frames):
    f = critic_forward(phi, s, a, keep, frames)
    e = f["q"] - np.asarray(y, np.float64)
    _f32(e, "q - y")
    _f32(e * e, "squared error")
    _rows_exact(np.ones((len(e), 1)), (e * e)[:, None], "sum of squared errors")
    d0 = 2.0 * e / ng
    _bf16_pair(d0, "dz3")
    _rows_exact(np.ones((len(e), 1)), d0[:, None], "db3")
    _rows_exact(f["h2"], d0[:, None], "dW3")
    dz2 = d0[:, None] * f["w3"][:, 0][None, :] * (f["z2"] > 0)
    _bf16_exact(dz2, "critic dz2")
    _rows_exact(f["xa"], dz2, "critic dW2")
    _rows_exact(np.ones((len(e), 1)), dz2, "critic db2")
    dx2 = _sum_exact(dz2, f["w2"][:H1].T, what="critic dx2")
    dz1 = dx2 * (f["x2"] > 0) * (1.0 / (1.0 - RATE))
    _bf16_exact(dz1, "critic dz1")
    _rows_exact(s, dz1, "critic dW1")
    _rows_exact(np.ones((len(e), 1)), dz1, "critic db1")


def check_actor_grad(theta, phi_pi, s, frames):
    fa = actor_forward(theta, s, frames, paired=True)
    fc = critic_forward(phi_pi, s, np.zeros((len(s), 2)), None, frames)
    _rows_exact(np.ones((len(s), 1)), fc["q"][:, None], "sum q")
    up = fc["up"]
    _bf16_pair(up, "actor dz3")
    _rows_exact(np.ones((len(s), 1)), up, "actor db3")
    _rows_exact(fa["h2"], up, "actor dW3")
    _f32(up[:, :1] * fa["w3"][:, 0][None, :], "actor dz2 terms")
    _f32(up[:, 1:] * fa["w3"][:, 1][None, :], "actor dz2 terms")
    dz2 = _sum_exact(up, fa["w3"].T, what="actor dz2") * (fa["z2"] > 0)
    _bf16_exact(dz2, "actor dz2")
    _rows_exact(fa["h1"], dz2, "actor dW2")
    _rows_exact(np.ones((len(s), 1)), dz2, "actor db2")
    dx2 = _sum_exact(dz2, fa["w2"].T, what="actor dx2")
    dz1 = dx2 * (fa["h1"] > 0)
    _bf16_exact(dz1, "actor dz1")
    _rows_exact(s, dz1, "actor dW1")
    _rows_exact(np.ones((len(s), 1)), dz1, "actor db1")


def check_targets(theta, phis, r, s2, done, frames):
    actor_forward(theta, s2, frames, paired=True)
    q = np.min([critic_forward(p, s2, np.zeros((len(s2), 2)), None, frames)["q"] for p in phis], axis=0)
    _f32(GAMMA * q, "gamma q")
    _f32(np.asarray(r, np.float64) + GAMMA * (1.0 - done) * q, "TD target")


def premise(frames, n):
    """Every check for one shape of the GPU tests: forwards, both critics' targets, the policy gradient, and the critic
    gradient under the injected and the Philox mask."""
    b = make(frames, n)
    actor_forward(b["theta_fwd"], b["s"], frames, paired=False)
    critic_forward(b["phi"], b["s"], b["a"], None, frames)
    check_targets(b["theta"], [b["phi"], b["phi2"]], b["r"], b["s2"], b["done"], frames)
    check_actor_grad(b["theta"], b["phi_pi"], b["s"], frames)
    for keep in (b["keep"], philox_keep(n)):
        check_critic_grad(b["phi"], b["s"], b["a"], targets(b, keep), keep, n_global(n), frames)
    return b
