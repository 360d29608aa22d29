"""The fused physics step (step_pp_kernel, one thread per player) streams each lane's actions through a ring of RING_SLOTS
slots in shared memory: a prologue fills all but one slot, every tick refills the slot of the tick before it, and ticks past
the end of the launch are zero-filled.  Launches of 2, RING_SLOTS - 1, RING_SLOTS, RING_SLOTS + 1 and 2 * RING_SLOTS + 1
ticks put the end of the launch on each side of the prologue and of one full turn of the ring, at every CTA size (the
ring's slot stride is the CTA size).

The launches must reach step_pp_kernel, which only physics-only steps do: parity.check_bench_shape steps with
want_obs=False and terminal reward, and compares every reward, done flag and winner of every tick and the state after every
launch with the oracle.  A 5-tick limit restarts games inside the launches, so the reset path (which re-turns from the
next tick's action) runs beside the ring as well."""
import pytest

from tests import parity

pytestmark = pytest.mark.gpu

RING_SLOTS = 8         # kRingD in skillshot_learning_b200/csrc/ss_env.cu


def make(n, **kw):
    from skillshot_learning_b200.game import SkillshotEnvs
    return SkillshotEnvs(n, device="cuda:0", **kw)


@pytest.mark.parametrize("blk", ["64", "448", "896"])
@pytest.mark.parametrize("chunk", [2, RING_SLOTS - 1, RING_SLOTS, RING_SLOTS + 1, 2 * RING_SLOTS + 1])
def test_fused_physics_ring_edges_match_oracle(monkeypatch, chunk, blk):
    monkeypatch.setenv("SS_STEP_BLK", blk)
    episodes, _ = parity.check_bench_shape(make, n=1000 + 37, T=3 * chunk, K=chunk, seed=40 + chunk, tick_limit=5)
    assert episodes >= 1037 * (3 * chunk // 5)              # every env restarted on every 5th tick
