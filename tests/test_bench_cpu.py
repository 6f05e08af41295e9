"""bench.py's host logic on a CPU box: the whole script runs against tests/fake_b200mpi.py (host memory,
gloo between rank processes, the oracle's reduction orders) for a world of 1 and a world of 2 -- the
parity bookkeeping over whole buffers, the contract line and its extra objects, exit codes, and the
deadline that prints a partial line instead of losing the run.  No kernel runs here; the GPU suite and
the bench itself on a B200 box cover the product."""
import json
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RANK = os.path.join(ROOT, "tests", "_bench_fake_rank.py")

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "e2e", "gpu_launches", "clocks", "roofline"]


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def run_bench(n, *args, timeout=420, extra_env=None):
    port = free_port()
    procs = []
    for r in range(n):
        env = dict(os.environ, PYTHONPATH=ROOT, OMP_NUM_THREADS="1")
        env.update(extra_env or {})
        if n > 1:
            env.update(RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(n), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        else:
            for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
                env.pop(k, None)
        procs.append(subprocess.Popen([sys.executable, RANK, "--gpus", str(n)] + list(args), env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT))
    outs = [p.communicate(timeout=timeout) for p in procs]
    return [(p.returncode, o, e) for p, (o, e) in zip(procs, outs)]


def contract_line(stdout):
    lines = [ln for ln in stdout.splitlines() if ln.startswith('{"metric')]
    assert len(lines) == 1, stdout[-2000:]
    return json.loads(lines[0])


def test_bench_world_of_1_contract_line():
    (rc, out, err), = run_bench(1, "--bytes", str(1 << 20), "--steps", "3", "--warmup", "3", "--cpu-sample-bytes", str(1 << 18))
    assert rc == 0, err[-3000:]
    d = contract_line(out)
    for k in REQUIRED:
        assert k in d, k
    assert d["n_gpus"] == 1 and d["metric"] == "allreduce_f32_sum_algbw" and d["higher_is_better"] is True
    assert d["parity_ok"] is True and all(d["parity"].values()), d["parity"]
    assert d["e2e"]["h2d_bytes_per_step"] == 1 << 20 and d["e2e"]["roofline"]["bound"] == "pcie"
    assert d["e2e_pageable"]["registered"]["ms_per_step"] > 0
    assert d["roofline"]["bound"] == "hbm" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["parity_ok"] is True
    assert d["config"]["workload"].startswith("Allreduce float32 sum")


def test_bench_world_of_2_parity_dict_and_secondary():
    res = run_bench(2, "--bytes", str(4 << 20), "--steps", "3", "--warmup", "3", "--no-nccl")
    assert all(rc == 0 for rc, _, _ in res), "\n".join(e[-2500:] for _, _, e in res)
    assert not any(ln.startswith('{"metric') for ln in res[1][1].splitlines()), "only rank 0 prints"
    d = contract_line(res[0][1])
    for k in REQUIRED + ["parity", "secondary", "e2e_pageable"]:
        assert k in d, k
    assert d["n_gpus"] == 2 and d["metric"] == "allreduce_f32_sum_busbw" and d["scaling"] == "weak"
    want = {"allreduce_f32_full_buffer", "allreduce_f32_odd_count_in_place", "allreduce_f32_64MiB_twoshot", "allreduce_f32_64MiB_twoshot_smem",
            "allreduce_f32_64MiB_ring", "allreduce_ll_small", "bcast_f32_root0", "bcast_f32_root1", "allgather_i64_1Mi_auto", "allgather_i64_1Mi_push",
            "allgather_i64_1Mi_ring", "reduce_scatter_i64", "bounce_f64_1MiB", "e2e_host_result", "e2e_pageable_result"}
    assert want <= set(d["parity"]), sorted(want - set(d["parity"]))
    assert d["parity_ok"] is True and all(d["parity"].values()), {k: v for k, v in d["parity"].items() if not v}
    sec = d["secondary"]
    assert sec["bcast_4MiB_busbw_gbs"] > 0 and sec["allgather_1Mi_i64_busbw_gbs"] > 0 and sec["bounce_1MiB_f64_rt_us_host"] > 0
    assert d["roofline"]["bound"] == "nvlink" and "nvlink_counters" in d["roofline"]
    assert set(sec["link_probe_gbs_per_direction"]) == {"rank0_pulls_other_direction_idle", "rank0_pushes_other_direction_idle", "all_ranks_pull",
                                                        "all_ranks_push", "all_ranks_pull_and_push"}
    assert d["e2e"]["frac_of_roofline"] > 0


def test_bench_world_of_2_switch_branches():
    """The same run with the fake claiming a multicast mapping: the NVLS / hybrid branches of the parity
    section (tolerance checks, their keys, restoring the hybrid parameter) execute."""
    res = run_bench(2, "--bytes", str(4 << 20), "--steps", "3", "--warmup", "3", "--no-nccl", "--no-e2e", "--no-secondary", extra_env={"FAKE_NVLS": "1"})
    assert all(rc == 0 for rc, _, _ in res), "\n".join(e[-2500:] for _, _, e in res)
    d = contract_line(res[0][1])
    want = {"allreduce_i64_nvls", "allreduce_f32_64MiB_nvls", "allreduce_f32_64MiB_hybrid", "allgather_i64_1Mi_nvls"}
    assert want <= set(d["parity"]), sorted(want - set(d["parity"]))
    assert d["parity_ok"] is True, {k: v for k, v in d["parity"].items() if not v}
    assert d["config"]["nvls"] is True and d["e2e"] is None


def test_bench_world_of_2_nccl_comparison_block():
    """The NCCL comparison block of bench.py (bound with ctypes on a GPU box) against a stand-in with the
    same five entry points: init, timing loops, the result cross-check against the oracle, no deadline hit."""
    res = run_bench(2, "--bytes", str(4 << 20), "--steps", "3", "--warmup", "3", "--no-parity", "--no-e2e", extra_env={"FAKE_NCCL": "1"})
    assert all(rc == 0 for rc, _, _ in res), "\n".join(e[-2500:] for _, _, e in res)
    d = contract_line(res[0][1])
    c = d["secondary"]["nccl_allreduce_comparison"]
    assert c["version"] == 22703 and set(c["sizes"]) == {"1024", "1048576", str(4 << 20)}, c
    assert c["result_agrees_with_oracle"] is True, c


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs: a world of 1 writes the whole result (a copy of its seeded input), the same on every
    run; a world of 2 above the size limit writes the documented seeded sample of the sum on each rank."""
    import numpy as np
    import bench
    from oracle import oracle as O
    count = (1 << 20) // 4
    for d in ("a", "b"):
        (rc, out, err), = run_bench(1, "--bytes", str(count * 4), "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-e2e",
                                    "--dump-outputs", str(tmp_path / d))
        assert rc == 0, err[-3000:]
    a, b = np.load(tmp_path / "a" / "allreduce_recv_rank0.npy"), np.load(tmp_path / "b" / "allreduce_recv_rank0.npy")
    assert a.dtype == np.float32 and np.array_equal(a, O.fill(np.float32, bench.SEED, count)) and np.array_equal(a, b)

    count = bench.DUMP_ELEMS + 3  # two ranks: a sample of every other element, seeded offsets, a tail left out
    res = run_bench(2, "--bytes", str(count * 4), "--steps", "2", "--warmup", "3", "--no-parity", "--no-e2e", "--no-secondary", "--no-nccl",
                    "--dump-outputs", str(tmp_path / "c"))
    assert all(rc == 0 for rc, _, _ in res), "\n".join(e[-2500:] for _, _, e in res)
    k = bench.DUMP_ELEMS // 2
    stride = count // k
    idx = np.arange(k) * stride + np.random.default_rng(bench.SEED).integers(0, stride, k)
    want = O.allreduce([O.fill(np.float32, bench.SEED + r, count) for r in range(2)])[idx]
    total = 0
    for r in range(2):
        got = np.load(tmp_path / "c" / ("allreduce_recv_rank%d.npy" % r))
        assert got.dtype == np.float32 and np.array_equal(got, want), r
        total += got.nbytes
    assert total <= 64 << 20
    rc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, cwd=ROOT).returncode
    assert rc == 2, "--steps 0 must be refused, not run zero timed steps"


def test_bench_deadline_prints_a_partial_line():
    """--deadline in the past: the sections after the timed region are cut short, rank 0 still prints
    the contract keys and every rank exits 0."""
    res = run_bench(2, "--bytes", str(4 << 20), "--steps", "3", "--warmup", "3", "--no-nccl", "--no-parity", "--deadline", "1",
                    extra_env={"FAKE_SLOW_PROBE_S": "6"})
    assert all(rc == 0 for rc, _, _ in res), "\n".join(e[-2500:] for _, _, e in res)
    d = contract_line(res[0][1])
    for k in REQUIRED:
        assert k in d, k
    assert "partial line" in d["config"]["note"] and d["value"] > 0
