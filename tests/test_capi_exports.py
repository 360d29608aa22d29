"""The C-ABI library loads and exports every symbol include/skillshot_b200.h declares
(no compute calls: this runs without a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ss_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from skillshot_learning_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared_symbols()
    assert "ss_env_step" in names and len(names) >= 8
    for n in names:
        assert hasattr(lib, n), n
        assert n in _lib.SIGNATURES, "binding missing for " + n
    assert lib.ss_version() >= 100
    lib.ss_state_bytes.restype = ctypes.c_int64
    assert lib.ss_state_bytes(ctypes.c_int64(10)) == 640


def test_invalid_arguments_are_rejected_without_a_gpu():
    from skillshot_learning_b200 import _lib
    assert _lib.lib.ss_env_reset(None, 4, None, 0, None, 0, 0, None) == -1
    assert _lib.lib.ss_env_step(None, 4, None, None, None, None, None, 1, 1, 0, 0, 0, 0, 0, None, None, 0, None) == -1


def test_learner_entry_points_reject_invalid_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L = _lib.lib
    assert L.ss_learner_workspace_bytes() >= 148 * (36609 + 1) * 4
    assert L.ss_actor_forward(None, None, None, 16, 0.0, 1, 0.0, 0, 0, None) == -1
    assert L.ss_actor_forward_tc(None, None, None, 16, 0.0, 1, 0.0, 0, 0, None) == -1
    assert L.ss_critic_forward(None, None, None, None, 16, None) == -1
    assert L.ss_critic_forward_tc(None, None, None, 16, None, None, None, None, 0.0, None, None) == -1
    assert L.ss_critic_grad(None, None, None, None, None, 0.2, 0, 0, 16, 16, 0, None, None, None, 0, None) == -1
    assert L.ss_critic_grad_tc(None, None, None, None, None, 0.2, 0, 0, 16, 16, 0, None, None, None, 0, None) == -1
    assert L.ss_actor_grad(None, None, None, 16, None, None, None, 0, None) == -1
    assert L.ss_actor_grad_tc(None, None, None, 16, None, None, None, 0, None) == -1
    assert L.ss_adam_tf(None, None, None, None, None, 10, 1, 1e-3, 0.9, 0.999, 1e-7, 1.0, 1.0, None) == -1
    assert L.ss_replay_push(None, None, None, None, None, 10, 0, None, None, None, None, None, 1, 4, None) == -1
    # flags | inbox[2][world][capacity] | the one-kernel exchange's flags [2][world][ceil((capacity + 1) / 64)]
    assert L.ss_peer_bytes(9, 100) == -1 and L.ss_peer_bytes(2, 100) == 256 + 2 * 2 * 100 * 4 + 2 * 2 * 2 * 4
    assert L.ss_peer_reduce_adam_tf(None, 1, 10, None, None, 2, 0, 100, 1, None, None, None, None, None, 1, 1e-3, 0.9, 0.999, 1e-7,
                                    1.0, 1.0, None, None) == -1
    assert L.ss_actor_critic_forward_tc(None, None, None, None, 16, None, None, None, None, 0.0, None, None, None) == -1
    assert L.ss_set_dependent_launch(-1) == -1
    assert L.ss_peer_reduce_push(None, 1, 10, None, None, 2, 0, 100, 1, None, None) == -1
    assert L.ss_ddpg_update(None, None) == -1
    assert L.ss_actor_frames_params(20) == 240 * 256 + 256 + 256 * 128 + 128 + 128 * 2 + 2 and L.ss_actor_frames_params(0) == -1
    assert L.ss_obs_stack_tc_bytes(131072, 20) == 1024 * 32 * 2048 and L.ss_obs_stack_tc_bytes(1, 1) == 2 * 2048
    assert L.ss_obs_stack_tc_bytes(16, 21) == -1
    assert L.ss_actor_frames_tc_workspace_bytes(131072, 1024) == 1024 * 65536 and L.ss_actor_frames_tc_workspace_bytes(300, 0) == 3 * 65536
    assert L.ss_obs_stack_push(None, 16, 20, 0, None, None, 1, None) == -1
    assert L.ss_obs_stack_push_tc(None, 16, 20, 0, None, None, 1, None) == -1
    assert L.ss_param_noise_groups(None, None, 100, 2, 100, 0.5, 0, 0, None) == -1
    assert L.ss_actor_forward_frames(None, 0, 0, None, 20, 0, None, 16, None) == -1
    assert L.ss_actor_forward_frames_tc(None, 0, 0, None, 20, 0, None, 16, None, 0, None) == -1
    blank = _lib.DdpgUpdateArgs()
    blank.batch, blank.size, blank.capacity, blank.step_actor, blank.step_critic = 16, 16, 16, 1, 1
    assert L.ss_ddpg_update(ctypes.byref(blank), None) == -1


def test_update_argument_block_matches_the_header():
    """The ctypes mirror of struct ss_ddpg_update_args lists the header's fields in the header's order."""
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    body = re.search(r"typedef struct ss_ddpg_update_args \{(.*?)\} ss_ddpg_update_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.sub(r"[\s\*]|const", "", part.split()[-1] if i else part.split()[-1])
                      for i, part in enumerate(decl.split(","))]
    assert names == [f[0] for f in _lib.DdpgUpdateArgs._fields_]


def test_product_package_does_not_touch_the_oracle():
    pkg = os.path.join(ROOT, "skillshot_learning_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle-free", ""), os.path.join(dirpath, f)
                assert "hostsim" not in src or f == "ss_env_core.cuh", os.path.join(dirpath, f)


def test_binding_arity_matches_the_header():
    """Every ctypes signature in _lib.SIGNATURES has as many parameters as the header's prototype."""
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"typedef struct.*?\}\s*\w+;", "", text, flags=re.S)
    protos = dict(re.findall(r"\b(ss_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S))
    assert len(protos) >= 40
    for name, params in protos.items():
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert name in _lib.SIGNATURES, name
        assert len(_lib.SIGNATURES[name][1]) == n, (name, len(_lib.SIGNATURES[name][1]), n)


def test_bench_report_assembles_without_a_gpu():
    """bench.py's learner report is plain arithmetic on the measured times: build it from made-up times for 1 and 8
    ranks so that a typo in a key or a format string shows up here and not at the end of a GPU run."""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    peaks = {"hbm_gbs": 6556.5, "bf16_tflops": 1631.0}
    times = dict(zip(bench.LEG_KEYS, (0.08, 0.19, 0.044, 2.1, 0.79, 0.094, 0.188, 0.49, 0.17, 0.52, 4.4)))
    for world, collective in ((1, "peer"), (8, "peer"), (2, "nccl")):
        rep = bench.learner_report(times, world, peaks, "measured", collective, dict(times, roll=0.079, cfg5=0.09))
        json.dumps(rep)
        want = {"rollout", "train", "selfplay_training", "planning_actor_speed_sweep", "actor_forward_roofline"}
        assert set(rep) == (want | {"scaling_in_run"} if world > 1 else want)
        assert rep["train"]["samples_per_sec"] == world * bench.TRAIN_BATCH / 0.19e-3
        assert 0 < rep["actor_forward_roofline"]["frac"] < 1
        if world > 1:
            sc = rep["scaling_in_run"]
            assert abs(sc["update_weak_efficiency"] - 0.17 / 0.19) < 1e-12
            assert abs(sc["config4_strong_efficiency"] - 0.52 / 0.49 / world) < 1e-12
    assert bench.ncu_traffic(bench.TICKS_PER_LAUNCH) is not None and bench.ncu_traffic(7) is None
    prof = bench.ncu_profile(bench.TICKS_PER_LAUNCH)
    assert prof["step_kernel_physics_warp_inst_per_launch"] > prof["step_kernel_physics_fp64_warp_inst_per_launch"] > 0
    # both arms print the same config object (the driver compares them)
    cfg = bench.bench_config(bench.TICKS, bench.TICKS_PER_LAUNCH)
    assert set(cfg) == {"workload", "envs_per_gpu", "ticks_per_step", "ticks_per_launch", "l2"}


def test_bench_dump_outputs_writes_a_seeded_float_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs on made-up step outputs: float32 / float64 files only, the byte bound on the step outputs
    held, the same env columns on every call, and the sampled values those of the step."""
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("_bench3", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_STEP_BYTES", 16 * 64 * 100)
    n, K = 1000, 64
    g = torch.Generator().manual_seed(0)
    out = dict(reward=torch.randn((K, n, 2), generator=g), done=torch.randint(0, 2, (K, n), generator=g, dtype=torch.uint8),
               winner=torch.randint(0, 3, (K, n), generator=g, dtype=torch.uint8))

    class Envs:
        n_envs = n

        def export_state(self):
            return dict(px=np.arange(2 * n, dtype=np.int64).reshape(n, 2), prot=np.full((n, 2), 0.5), ticks=np.arange(n))

    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), Envs(), out)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    step_bytes = 0
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
        step_bytes += a.nbytes if f in ("reward.npy", "done.npy", "winner.npy") else 0
    assert step_bytes <= bench.DUMP_STEP_BYTES
    cols = np.load(tmp_path / "a" / "env_index.npy").astype(np.int64)
    assert len(cols) == 100 and np.all(np.diff(cols) > 0)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "reward.npy"), out["reward"].numpy()[:, cols])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "winner.npy"), out["winner"].numpy()[:, cols])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "state_px.npy"), Envs().export_state()["px"])


def test_cpu_legs_ignore_omp_num_threads(monkeypatch):
    """torch.distributed.run exports OMP_NUM_THREADS=1: the CPU legs size themselves from the CPU affinity instead."""
    import importlib.util
    monkeypatch.setenv("OMP_NUM_THREADS", "1")
    spec = importlib.util.spec_from_file_location("_bench2", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.host_cores() == len(os.sched_getaffinity(0))
    if bench.host_cores() > 1:
        from oracle.oracle import lib as olib
        dt, envs, actions = bench.cpu_port_run(4096, 4, bench.host_cores())
        assert olib().ss_oracle_max_threads() == bench.host_cores()      # omp_set_num_threads took effect


def test_header_constants_match_the_python_mirror():
    """SS_PAIR_MAIL_EMPTY (the empty mark of ss_actor_critic_forward_tc's mailbox) and the status bits are written twice, in
    include/skillshot_b200.h and in _lib.py: they must agree."""
    import re
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    m = re.search(r"#define\s+SS_PAIR_MAIL_EMPTY\s+(0x[0-9a-fA-F]+)", text)
    assert m and int(m.group(1), 16) == _lib.PAIR_MAIL_EMPTY
    m = re.search(r"#define\s+SS_STATUS_ROLLOUT_TIMEOUT\s+(\d+)", text)
    assert m and int(m.group(1)) == 4


def test_public_header_is_plain_c(tmp_path):
    """include/skillshot_b200.h is the drop-in boundary: it must compile as C99 on its own (no C++ or CUDA types in the
    signatures), with every struct complete."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "hdr.c"
    src.write_text('#include "skillshot_b200.h"\n'
                   'int main(void) { ss_ddpg_update_args a; (void)a; return SS_PAIR_MAIL_EMPTY == 0x7fc0dead ? 0 : 1; }\n')
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                    "-o", str(tmp_path / "hdr.o")], check=True)
