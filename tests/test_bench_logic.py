"""Host logic of bench.py that must hold on every rank count: loops that contain collectives run the same number of
iterations on all ranks (a per-rank clock deadlocked an 8-GPU run once), and the reference arm prints the contract's
JSON line without touching the GPU."""
import json
import os
import socket
import subprocess
import sys
import time

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import bench
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    buf = [torch.zeros(4) for _ in range(world)]
    calls = [0]

    def step():                                   # a step with a collective in it; rank 1 is 5x slower than rank 0
        time.sleep(0.002 if rank == 0 else 0.010)
        dist.all_gather(buf, torch.full((4,), float(rank)))
        calls[0] += 1

    def reduce_max(flags):
        t = torch.tensor(flags, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    t0 = time.perf_counter()

    def stop_flags():                             # per-rank opinions differ: rank 0 is "stable" early, rank 1 never is
        el = time.perf_counter() - t0
        return (rank == 0 and el > 0.05), el > (0.25 if rank == 0 else 0.30)

    n, secs = bench.collective_preheat(step, lambda: None, stop_flags, world, reduce_max)
    for _ in range(3):                            # "warm-up + timed" steps afterwards must still pair up
        step()
    dist.barrier()
    with open(os.path.join(out_dir, f"r{rank}.json"), "w") as f:
        json.dump({"n": n, "calls": calls[0]}, f)
    dist.destroy_process_group()


def test_preheat_runs_the_same_number_of_collective_steps_on_every_rank(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r = [json.load(open(tmp_path / f"r{i}.json")) for i in range(world)]
    assert r[0] == r[1] and r[0]["n"] >= 4 and r[0]["calls"] == r[0]["n"] + 3


def test_preheat_single_rank_stops_on_stable_or_timeout():
    sys.path.insert(0, ROOT)
    import bench
    calls = [0]

    def step():
        calls[0] += 1
        time.sleep(0.001)
    n, _ = bench.collective_preheat(step, lambda: None, lambda: (True, False), 1)
    assert n == calls[0] == 4                                             # stable at once: one chunk
    t0 = time.perf_counter()
    n, secs = bench.collective_preheat(step, lambda: None, lambda: (False, time.perf_counter() - t0 > 0.05), 1)
    assert n % 4 == 0 and n >= 8 and secs >= 0.05                         # never stable: runs into the time limit


def test_step_size_estimate_ignores_one_time_costs():
    """The batches-per-step estimate must come from settled batches: a slow first call (NCCL connection set-up took 0.3 s
    once and produced a 0.06 s 'timed region' at N = 8) may not leak into it."""
    sys.path.insert(0, ROOT)
    import bench

    class Sampler:
        def stable(self):
            return True
    calls = [0]

    def step():
        calls[0] += 1
        time.sleep(0.25 if calls[0] == 1 else 0.002)
    inner, ph_s, n_ph, est = bench.settle_and_estimate(step, lambda: None, lambda: None, Sampler(), 1, None, steps=10,
                                                       min_timed_s=0.5, preheat_max=0.4, settle_s=0.1)
    assert est < 0.01 and 15 <= inner <= 30            # ~2.2 ms per batch -> ~23 batches per step, not 1
    assert n_ph >= 4 and ph_s < 0.5


def test_host_data_pool_generates_canonical_chunks_and_the_parallel_oracle_equals_the_definition():
    """bench.py's worker pool: (i) what it writes into the shared mapping IS oracle.synth_rows chunk by chunk, also when a
    shard boundary cuts a chunk; (ii) its parallel oracle (per-piece fp32 prefilter + float64 re-scoring) returns exactly
    what the oracle's definition returns."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from oracle import bruteforce as bf
    old = bench.CHUNK
    bench.CHUNK = 1000                                                    # small chunks keep this a CPU-seconds test
    try:
        dim, n_total, lo, hi = 64, 3500, 700, 3500                        # rows 700..3499: cuts chunk 0, ragged last chunk
        host = bench.HostData((hi - lo) * dim * 2, 3)
        seen = []
        host.generate(77, dim, lo, hi, n_total, lambda first, n: seen.append((first, n)))
        shard = host.view(hi - lo, dim).copy()
        want = np.concatenate([bf.synth_rows(77, c, min(1000, n_total - c * 1000), dim) for c in range(4)])[lo:hi]
        assert (shard == want).all() and sorted(seen) == [(0, 300), (300, 1000), (1300, 1000), (2300, 500)]
        q = bf.synth_queries(78, 9, dim, want[:1000])
        rs, ri = host.oracle_topk(q, hi - lo, dim, 10)
        host.close()
        es, ei = bf.cosine_topk_f64(q, want, 10)
        assert (ri == ei).all() and np.abs(rs - es).max() < 1e-15
    finally:
        bench.CHUNK = old


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample-queries", "8", "--cpu-sample-rows", "4096", "--gpus", "1"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["config"]["workload"].startswith("10000000x1536")
    # other ranks of a torchrun launch print nothing and exit 0
    out1 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                          capture_output=True, text=True, env=dict(env, RANK="1", WORLD_SIZE="2"), timeout=120)
    assert out1.returncode == 0 and out1.stdout.strip() == ""


def test_dump_outputs_saves_the_answer_as_float_arrays(tmp_path):
    """--dump-outputs: what search() returned, scores as float32 and corpus rows as float64 holding the exact rows."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    s = torch.tensor([[0.75, 0.5], [1.0, -1.0]], dtype=torch.float32)
    i = torch.tensor([[9_999_999, 0], [3, 2**31 - 1]], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "out"), (s, i))
    scores, indices = np.load(tmp_path / "out" / "scores.npy"), np.load(tmp_path / "out" / "indices.npy")
    assert scores.dtype == np.float32 and (scores == s.numpy()).all()
    assert indices.dtype == np.float64 and (indices == i.numpy()).all()
    assert sorted(os.listdir(tmp_path / "out")) == ["indices.npy", "scores.npy"]


def test_bench_rejects_arguments_it_cannot_honour(tmp_path):
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and out.stdout == "", args


def test_harness_and_tool_scripts_compile():
    """The GPU harness can only run on a B200 box; at least keep it syntactically alive here."""
    import glob
    import py_compile
    files = glob.glob(os.path.join(ROOT, "tools", "*.py")) + glob.glob(os.path.join(ROOT, "tests", "harness", "*.py")) + \
        [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]
    assert len(files) >= 8
    for f in files:
        py_compile.compile(f, doraise=True)
    for sh in glob.glob(os.path.join(ROOT, "tools", "*.sh")):
        assert subprocess.run(["bash", "-n", sh]).returncode == 0, sh
        for ref in __import__("re").findall(r"(?:python|bash) ((?:tools|tests)/[\w/.]+)", open(sh).read()):
            assert os.path.exists(os.path.join(ROOT, ref)), f"{sh} refers to missing {ref}"
