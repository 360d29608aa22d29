"""Launch time of the fused physics step (ss_env_step, terminal reward, no observations: bench.py's timed kernel) for
several builds of the library in one process, alternated.

    python tools/step_ring_time.py --lib stock=/path/a.so --lib ring=/path/b.so [--reps 7] [--shapes 65536x1024,...]

Each library is loaded on its own (ctypes, RTLD_LOCAL) and gets its own env state, reset from the same seed; all of them
read the same action buffers.  Per shape and library, 20 launches are captured in a CUDA graph; one sample is the mean
launch time over enough replays to fill ~0.25 s, timed with CUDA events.  The libraries take turns sample by sample, so a
drift of the clocks or a neighbour on the machine lands on all of them alike.  The action buffers of a shape rotate over
more than the 126 MB of L2 where memory allows (as tools/explore_step.py does).  After timing, each library's outputs of
its last launch and its env state are compared with the first library's: equal numbers of identical launches from equal
states must give equal bytes when the kernels compute the same thing.

Prints the card, its power limit and SM clocks, then one line per shape and library: median, min and max microseconds per
launch, env-steps/s at the median and the median's ratio to the first library's."""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from skillshot_learning_b200 import _lib

PER_GRAPH = 20
DEFAULT_SHAPES = "65536x32,65536x256,65536x1024,262144x256,1048576x256"


def card() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def load(path: str) -> ctypes.CDLL:
    lib = ctypes.CDLL(os.path.abspath(path))
    for name in ("ss_state_bytes", "ss_env_reset", "ss_env_step"):
        res, args = _lib.SIGNATURES[name]
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


class Arm:
    """One library at one shape: its state, outputs and the captured graph."""

    def __init__(self, lib, E, K, acts, stream):
        self.lib, self.E, self.K = lib, E, K
        self.state = torch.zeros(lib.ss_state_bytes(E), dtype=torch.uint8, device="cuda")
        self.reward = torch.zeros((K, E, 2), dtype=torch.float32, device="cuda")
        self.done = torch.zeros((K, E), dtype=torch.uint8, device="cuda")
        self.winner = torch.zeros((K, E), dtype=torch.uint8, device="cuda")
        self.status = torch.zeros(32, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()            # the buffers (and the actions) were written on the default stream
        with torch.cuda.stream(stream):
            self.check(lib.ss_env_reset(self.state.data_ptr(), E, None, _lib.RESET_RANDOM, None, 1, 0, stream.cuda_stream))
            for j in range(3):
                self.launch(acts[j % len(acts)], 1 + j * K, stream)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=stream):
                for j in range(PER_GRAPH):
                    self.launch(acts[j % len(acts)], 1 + (3 + j) * K, stream)
        torch.cuda.synchronize()

    @staticmethod
    def check(rc):
        if rc != 0:
            raise RuntimeError("library call failed with code %d" % rc)

    def launch(self, a, counter, stream):
        self.check(self.lib.ss_env_step(self.state.data_ptr(), self.E, a.data_ptr(), None, self.reward.data_ptr(),
                                        self.done.data_ptr(), self.winner.data_ptr(), self.K, _lib.REWARD_TERMINAL, 2000, 1,
                                        _lib.RESET_RANDOM, 1, counter, None, self.status.data_ptr(), 0, stream.cuda_stream))

    def sample(self, replays, stream) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(replays):
                self.graph.replay()
            e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (replays * PER_GRAPH)

    def outputs(self):
        return (self.reward, self.done, self.winner, self.state, self.status)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, metavar="NAME=PATH")
    ap.add_argument("--shapes", default=DEFAULT_SHAPES, help="envs x ticks per launch, comma separated")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    libs = [(s.split("=", 1)[0], load(s.split("=", 1)[1])) for s in args.lib]
    print("card:", card(), flush=True)
    print("shape lib median_us min_us max_us env_steps_per_s ratio_to_%s outputs_equal" % libs[0][0], flush=True)
    stream = torch.cuda.Stream()
    for shape in args.shapes.split(","):
        E, K = (int(x) for x in shape.split("x"))
        g = torch.Generator(device="cuda").manual_seed(5)
        nbuf = max(1, min(PER_GRAPH, int(4e8 // (E * K * 16))))
        acts = [(torch.rand((K, E, 2, 2), device="cuda", generator=g) * 2.4 - 1.2).contiguous() for _ in range(nbuf)]
        arms = [Arm(lib, E, K, acts, stream) for _, lib in libs]
        t1 = arms[0].sample(1, stream)
        replays = max(2, int(0.25e6 / (t1 * PER_GRAPH)))
        for a in arms[1:]:
            a.sample(1, stream)
        times = [[] for _ in arms]
        for r in range(args.reps):
            order = range(len(arms)) if r % 2 == 0 else reversed(range(len(arms)))
            for i in order:
                times[i].append(arms[i].sample(replays, stream))
        med0 = statistics.median(times[0])
        ref = arms[0].outputs()
        for (name, _), a, ts in zip(libs, arms, times):
            same = all(torch.equal(x, y) for x, y in zip(ref, a.outputs()))
            m = statistics.median(ts)
            print("%s %s %.2f %.2f %.2f %.3e %.4f %s" % (shape, name, m, min(ts), max(ts), E * K / (m * 1e-6), m / med0,
                                                         "yes" if same else "no"), flush=True)
        del arms, acts
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
