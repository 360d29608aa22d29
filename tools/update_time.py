"""Development: device time of one DDPG update (the bench's update leg) at a few minibatch sizes."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from skillshot_learning_b200 import SelfPlayTrainer
E = 262144
for batch in [int(x) for x in (sys.argv[1:] or ["65536", "524288"])]:
    tr = SelfPlayTrainer(E, device="cuda:0", seed=0, replay_capacity=2 * E * 4, batch_size=batch, gamma=0.99, tau=0.005, precision="bf16",
                         noise_group=4096, tick_limit=200)
    tr.rollout(4)
    for _ in range(20):
        tr.update()
    torch.cuda.synchronize()
    best = 1e9
    for rep in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(200):
            tr.update()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / 200 * 1e3)
    print("batch %7d  update %.1f us  (sse %.6g  q %.6g)" % (batch, best, float(tr.networks.stats[0]), float(tr.networks.stats[1])),
          flush=True)
    del tr
