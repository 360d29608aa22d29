"""TD3 target and update restated with torch autograd on top of oracle/learner_oracle.py (no reference code; DESIGN.md
section 6.14).  Test infrastructure: tests/test_gpu_td3.py compares ActorCritic.td3_step and the ss_td3_targets* entry
points with it, every random choice (smoothing normals, dropout masks) injected."""
import numpy as np
import torch

from oracle.learner_oracle import AdamTF, actor_forward, actor_grad, critic_forward, critic_grad, soft_update


def td3_targets(theta_t, phi_t, phi2_t, r, s2, done, gamma, eps=None, sigma=0.0, clip=0.5, dtype=torch.float32):
    """y = r + gamma (1 - done) min(Q1'(s2, a~), Q2'(s2, a~)),  a~ = clamp(mu'(s2) + clamp(sigma eps, -clip, clip), -1, 1).
    phi2_t None: one critic; eps [n, 2]: the smoothing normals (injected), unused when sigma = 0.  Float32 arithmetic in the
    order of the library's epilogue."""
    r = np.asarray(r, np.float32)
    if gamma == 0.0:
        return r.copy()
    a2 = actor_forward(theta_t, s2, dtype).astype(np.float32)
    if sigma > 0.0:
        noise = np.clip(np.float32(sigma) * np.asarray(eps, np.float32), np.float32(-clip), np.float32(clip))
        a2 = np.clip(a2 + noise, np.float32(-1.0), np.float32(1.0)).astype(np.float32)
    q = critic_forward(phi_t, s2, a2, None, dtype=dtype)
    if phi2_t is not None:
        q = np.minimum(q, critic_forward(phi2_t, s2, a2, None, dtype=dtype))
    return (r + np.float32(gamma) * (1.0 - np.asarray(done, np.float32)) * q).astype(np.float32)


class TD3Oracle:
    """The TD3 update of ActorCritic.td3_step with every random choice injected: the target, a critic step on critic 1
    and one on critic 2 against the same y, and on every policy_delay-th update the actor step against critic 1 and the
    soft update of every target network (tau = 0 on the others)."""

    def __init__(self, theta, phi, phi2=None, gamma=0.99, tau=0.005, policy_delay=2, sigma=0.2, clip=0.5, dropout=0.2):
        self.theta, self.phi = np.asarray(theta, np.float32).copy(), np.asarray(phi, np.float32).copy()
        self.phi2 = None if phi2 is None else np.asarray(phi2, np.float32).copy()
        self.theta_t, self.phi_t = self.theta.copy(), self.phi.copy()
        self.phi2_t = None if phi2 is None else self.phi2.copy()
        self.opt_actor, self.opt_critic = AdamTF(self.theta.size), AdamTF(self.phi.size)
        self.opt_critic2 = None if phi2 is None else AdamTF(self.phi.size)
        self.gamma, self.tau, self.policy_delay, self.sigma, self.clip, self.dropout = gamma, tau, policy_delay, sigma, clip, dropout
        self.updates = 0

    def update(self, s, a, r, s2, done, eps, keep1, keep2=None):
        """eps [n, 2]: the smoothing normals; keep1 / keep2: the two critic steps' dropout masks [n, 256]."""
        y = td3_targets(self.theta_t, self.phi_t, self.phi2_t, r, s2, done, self.gamma, eps, self.sigma, self.clip)
        delayed = (self.updates + 1) % self.policy_delay == 0
        tau = self.tau if delayed else 0.0
        g, _ = critic_grad(self.phi, s, a, y, keep1, self.dropout)
        self.phi = self.opt_critic.step(self.phi, g)
        self.phi_t = soft_update(self.phi_t, self.phi, tau)
        if self.phi2 is not None:
            g, _ = critic_grad(self.phi2, s, a, y, keep2, self.dropout)
            self.phi2 = self.opt_critic2.step(self.phi2, g)
            self.phi2_t = soft_update(self.phi2_t, self.phi2, tau)
        if delayed:
            g, _ = actor_grad(self.theta, self.phi, s)
            self.theta = self.opt_actor.step(self.theta, g)
            self.theta_t = soft_update(self.theta_t, self.theta, tau)
        self.updates += 1
        return y
