"""CPU-side checks of bench.py's plumbing: the one-JSON-line contract survives a sub-record that hangs or raises,
the reference arm prints the keys of the result line (it is the CPU path, so it runs here), and --dump-outputs writes
exact, bounded, reproducible files."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_py(code, timeout=60):
    return subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=timeout)


def test_line_printed_once_on_the_normal_path():
    r = run_py("import bench\n"
               "e = bench.LineEmitter(0, {'value': 1})\n"
               "e.arm(30, 'late')\n"
               "e.finish(); e.finish()\n")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0]) == {"value": 1}


def test_watchdog_prints_the_headline_when_sub_records_hang():
    r = run_py("import bench, time\n"
               "e = bench.LineEmitter(0, {'value': 2})\n"
               "e.arm(0.3, 'sub-records stalled')\n"
               "time.sleep(30)\n"
               "print('not reached')\n")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    assert json.loads(lines[0]) == {"value": 2, "extra": {"error": "sub-records stalled"}}


def test_other_ranks_leave_silently():
    r = run_py("import bench\n"
               "e = bench.LineEmitter(3, None)\n"
               "e.abort('peer failed')\n"
               "print('not reached')\n")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_line():
    """`bench.py --impl reference` on a tiny sample: the reference's own CPU path (oracle/_ref, else the port)."""
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "64"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GCUPS" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["metric"].startswith("GCUPS")

    # a non-zero rank of the reference arm does no work and prints nothing
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, capture_output=True, text=True, timeout=60, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_exact_seeded_and_bounded(tmp_path):
    """--dump-outputs at the headline's 10^6 pairs: the kept pairs' record fields and op words exactly (op words above
    2^31 included), the same sample on every run, float64 files of under 64 MB in all."""
    import numpy as np
    import torch
    import bench
    from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
    n, stride = 1_000_000, 20
    items = torch.arange(n * 10, dtype=torch.int32)
    words = (np.arange(n * stride, dtype=np.uint64) * 2654435761 % 2 ** 32).astype(np.uint32)
    ops = torch.from_numpy(words.view(np.int32))
    for run in ("a", "b"):
        bench.write_outputs(str(tmp_path / run), bench.snapshot_outputs(torch, items, ops, n, stride, 1), n, 0, 1, None)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(["pair_index.npy", "ops.npy"] + [f + ".npy" for f in ITEM_DTYPE.names])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) < 64_000_000
    got = {f: np.load(tmp_path / "a" / f) for f in names}
    for f in names:
        assert got[f].dtype == np.float64 and np.array_equal(got[f], np.load(tmp_path / "b" / f))
    idx = got["pair_index.npy"].astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    for c, f in enumerate(ITEM_DTYPE.names):
        assert np.array_equal(got[f + ".npy"], idx * 10 + c)
    assert np.array_equal(got["ops.npy"], words.reshape(n, stride)[idx].astype(np.float64))
    assert got["ops.npy"].max() >= 2 ** 31

    # the reference arm has no GPU results: the combination is refused before any work
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--dump-outputs",
                        str(tmp_path / "ref")], cwd=ROOT, capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not os.path.exists(tmp_path / "ref")


def _dump_worker(rank, world, port, path):
    import numpy as np
    import torch
    import torch.distributed as dist
    import bench
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n, stride = 1000, 20
    items = torch.arange(n * 10, dtype=torch.int32) + 100_000 * rank       # stand-in for this rank's results
    ops = torch.from_numpy(np.full(n * stride, rank + 1, dtype=np.int32))
    bench.write_outputs(path, bench.snapshot_outputs(torch, items, ops, n, stride, world), n, rank, world, dist)
    dist.barrier()
    dist.destroy_process_group()


def test_dump_outputs_gathers_every_rank(tmp_path):
    """Several ranks: rank 0 writes DIR/<name>.npy with every rank's pairs, rank r's pair i at pair_index r * n + i."""
    import multiprocessing as mp
    import socket
    import numpy as np
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_dump_worker, args=(r, 2, port, str(tmp_path))) for r in range(2)]
    [p.start() for p in procs]
    [p.join(timeout=120) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    idx = np.load(tmp_path / "pair_index.npy")
    assert np.array_equal(idx, np.arange(2000))
    assert np.array_equal(np.load(tmp_path / "score.npy"), (idx % 1000) * 10 + 3 + 100_000 * (idx // 1000))
    assert np.array_equal(np.load(tmp_path / "ops.npy")[:, 0], 1 + idx // 1000)
