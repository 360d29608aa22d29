"""The premise of tests/test_gpu_learner_exact.py, checked without a GPU: on the networks and batches of tests/exact_nets.py
every operand the tensor-core kernels round is representable, every fp32 sum is exact in any order and no ReLU sits at 0 --
at every shape the GPU tests use.  If this passes and a GPU comparison there fails, the kernel is wrong."""
import numpy as np
import pytest

from tests import exact_nets as xn

SHAPES = sorted({(1, n) for n in xn.ROWS_12} | {(f, n) for f in range(1, 21) for n in xn.ROWS_FRAMES} |
                {(f, xn.ROWS_LARGE) for f in xn.FRAMES_LARGE} | {(f, n) for f, n, _ in xn.SHARDS})


@pytest.mark.parametrize("frames,n", SHAPES)
def test_every_rounding_is_exact(frames, n):
    xn.premise(frames, n)


def test_the_premise_check_rejects_inexact_inputs():
    """The checks are not vacuous: an action whose low half needs more than bf16, a loss divisor that is not a power of two,
    and biases on the integer grid (a unit sits at 0) are each rejected."""
    b = xn.make(1, 300)
    a = b["a"].copy()
    a[xn.fine_rows(300)[0], 0] = 0.5 + 2.0 ** -9 + 2.0 ** -18
    with pytest.raises(AssertionError, match="actions as a bf16 hi"):
        xn.critic_forward(b["phi"], b["s"], a, None, 1)
    with pytest.raises(AssertionError, match="dz3 in float32"):
        xn.check_critic_grad(b["phi"], b["s"], b["a"], xn.targets(b, b["keep"]), b["keep"], 300, 1)
    phi = b["phi"].copy()
    phi[12 * 256:13 * 256] = np.round(phi[12 * 256:13 * 256])            # b1 on the integer grid
    with pytest.raises(AssertionError, match="is 0"):
        xn.critic_forward(phi, b["s"], b["a"], None, 1)
