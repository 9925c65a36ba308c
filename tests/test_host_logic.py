"""Host-side logic: layout helpers, synthetic generator, sharding arithmetic, world_size-2 gather
over gloo.  CPU only."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from poseestimationkf_b200 import batched as B
from poseestimationkf_b200 import sharding as SH
from poseestimationkf_b200.synth import make_imu


def test_tri_full_roundtrip():
    A = torch.randn(5, 4, 4)
    P = A @ A.transpose(1, 2)
    tri = B.tri_from_full(P)
    assert tri.shape == (10, 5)
    torch.testing.assert_close(B.full_from_tri(tri), P)
    x = torch.arange(12.0).reshape(3, 4)
    torch.testing.assert_close(B.aos(B.soa(x)), x)


def test_initial_state_matches_reference_defaults():
    st = B.ReplayState.initial(3, "cpu", r=0.1, with_lpf=True)
    assert st.x.t().tolist() == [[1.0, 0.0, 0.0, 0.0]] * 3           # main_file.py:26
    torch.testing.assert_close(st.covariance(), torch.eye(4).expand(3, 4, 4))   # main_file.py:23
    torch.testing.assert_close(st.p[[0, 4, 7, 9]], torch.full((4, 3), 10.0))     # stored in units of r
    assert st.lpf.abs().sum() == 0                                    # KalmanFilter.cpp:16-18


def test_synth_properties():
    imu = make_imu(64, 300, seed=5, sigma=0.01, keep_truth=True)
    S = imu.streams
    assert S.shape == (300, 9, 64) and S.dtype == torch.float32
    for sl in (slice(3, 6), slice(6, 9)):
        n = torch.linalg.vector_norm(S[:, sl].double(), dim=1)
        assert (n - 1).abs().max() < 1e-6
    az0 = imu.acc_ref[2].abs()
    assert az0.min() > 0.02 and az0.max() < 0.98
    # deterministic in the seed, different across seeds
    again = make_imu(64, 300, seed=5, sigma=0.01)
    assert torch.equal(again.streams, S)
    assert not torch.equal(make_imu(64, 300, seed=6, sigma=0.01).streams, S)
    # measurements are the references seen through the true attitude: ref ~= R(q) meas
    q = imu.q_true[-1].T.numpy()
    w, x, y, z = q.T
    R = np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
                  np.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], -1),
                  np.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1)], 1)
    back = np.einsum("nij,nj->ni", R, S[-1, 3:6].T.double().numpy())
    assert np.abs(back - imu.acc_ref.T.double().numpy()).max() < 0.08     # sigma = 0.01 noise on both ends


def test_shard_bounds_cover_and_align():
    for n in (0, 1, 127, 128, 129, 1000, 1 << 20, 16777216, 16777216 + 5):
        for world in (1, 2, 3, 4, 8):
            spans = [SH.shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for (b0, e0), (b1, e1) in zip(spans, spans[1:]):
                assert e0 == b1 and b0 <= e0
            assert all(b % SH.ALIGN == 0 for b, _ in spans if b < n)
            sizes = SH.shard_sizes(n, world)
            assert sum(sizes) == n and max(sizes) - min(sizes) < 2 * SH.ALIGN
    assert SH.shard_sizes(16777216, 8) == [2097152] * 8


def test_time_chunks():
    assert list(SH.time_chunks(10, 4)) == [(0, 4), (4, 8), (8, 10)]
    assert list(SH.time_chunks(0, 4)) == []
    assert SH.chunk_steps_for_budget(1 << 20, 8 << 30) == (8 << 30) // ((1 << 20) * 36)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, n, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        b, e = SH.shard_bounds(n, rank, world)
        full = torch.arange(4 * n, dtype=torch.float32).reshape(4, n)
        got = SH.gather_states(full[:, b:e].contiguous(), n)
        slow = SH.max_over_ranks(float(rank + 1), "cpu")
        torch.save({"ok": torch.equal(got, full), "slow": slow}, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_gather_states_world2_gloo(tmp_path):
    world, n = 2, 1000            # ragged: 1000 = 7*128 + 104 -> shards of 512 and 488
    mp.spawn(_gather_worker, args=(world, _free_port(), n, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        res = torch.load(os.path.join(str(tmp_path), f"r{r}.pt"))
        assert res["ok"] and res["slow"] == 2.0


def test_log_reader_matches_the_reference_reader():
    """tests/golden/sample_log.txt was parsed by the reference's own ReadFile.getData (make_golden.py);
    logio.read_log must give exactly the same lists, and write_log must reproduce the file."""
    from poseestimationkf_b200 import compat, logio
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "log_parsed.npz"))
    path = os.path.join(os.path.dirname(__file__), "golden", "sample_log.txt")
    d = logio.read_log(path)
    for name in ("mag_0", "mag_1", "acc_0", "acc_1", "gyro", "timestamp", "quart_wahba", "quart_xk", "quart_gyro"):
        np.testing.assert_array_equal(np.asarray(getattr(d, name)), gold[name], err_msg=name)
    assert len(d.timestamp) == d.n_steps() + 1 and len(d.quart_xk) == d.n_steps() + 1      # T0 and the initial lines
    # the writer regenerates the file byte for byte from the parsed content
    lines = logio.format_log(acc_0=d.acc_0, mag_0=d.mag_0, t0_ns=d.timestamp[0][0], t_ns=[t[0] for t in d.timestamp[1:]],
                             gyro=d.gyro, mag_1=d.mag_1, acc_1=d.acc_1, x_k=d.quart_xk[1:], wahba_quart=d.quart_wahba[1:],
                             q_gyro=d.quart_gyro[1:])
    assert lines == open(path).read().splitlines()
    # compat module with the reference's class name
    sys.path.insert(0, compat.PATH)
    try:
        from ReadFile import getData
        g = getData(path)
        assert g.acc_1 == d.acc_1 and g.timestamp == d.timestamp and g.getArray("x : 1,2", 2) == [1.0, 2.0]
    finally:
        sys.path.remove(compat.PATH)
        sys.modules.pop("ReadFile", None)
    streams, acc_ref, mag_ref, dt = d.to_streams(device="cpu")
    assert streams.shape == (d.n_steps(), 9, 1) and dt.shape == (d.n_steps(),)
    np.testing.assert_allclose(dt.numpy(), 0.01, rtol=1e-6)
    np.testing.assert_allclose(streams[:, 3:6, 0].numpy(), np.asarray(d.acc_1), rtol=1e-6)


def test_cpulist_parsing_and_numa_binding_without_gpu():
    from poseestimationkf_b200 import sharding as SH
    assert SH._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert SH._parse_cpulist("") == set()
    # no CUDA device / no sysfs topology: binding is a no-op that says so
    import torch
    if not torch.cuda.is_available():
        assert SH.bind_host_to_gpu(0) is None


def test_reference_arm_contract_under_torchrun_world2():
    """`bench.py --impl reference` launched like our arm (torchrun, N = 2): rank 0 alone times the reference's CPU
    path and prints ONE JSON line with the contract's keys; the other rank exits 0 without output."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
           "--warmup", "1", "--cpu-seconds", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ekf_filter_steps_per_s" and d["unit"] == "filter-steps/s"
    assert d["n_gpus"] == 2 and d["higher_is_better"] is True and d["value"] > 0
    # the unmodified reference classes where their tree is present (this container), the oracle's port of them elsewhere (GPU box)
    import bench
    assert d["cpu_baseline"]["kind"] == ("reference" if bench.find_reference() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "configs[4]" in d["config"]["workload"] and d["scaling"] == "strong"      # 2 ranks: the sharded scaling run
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_sweep_partition_keeps_cells_and_stream_columns():
    """The per-cell precision split of a (Q,R) sweep: a partition of all filters into whole cells, original order kept,
    so that filter k of either group still reads stream column k % Ns."""
    Ns = 8
    grid = [(1e-3, 1e3), (1.0, 0.1), (1e3, 1e-3), (1.0, 1.0), (1e-2, 10.0), (10.0, 1e-2), (1.0, 99.0), (1.0, 100.0)]
    q = torch.tensor([q for q, _ in grid], dtype=torch.float32).repeat_interleave(Ns)
    r = torch.tensor([r for _, r in grid], dtype=torch.float32).repeat_interleave(Ns)
    plain, precise = B.sweep_partition(q, r, Ns)
    want = [bool(rr >= 100 * qq or qq >= 1e4 * rr) for qq, rr in grid]
    assert precise.numel() == Ns * sum(want) and plain.numel() == Ns * (len(grid) - sum(want))
    assert sorted(torch.cat([plain, precise]).tolist()) == list(range(len(grid) * Ns))
    for idx, flag in ((plain, False), (precise, True)):
        assert torch.equal(idx % Ns, torch.arange(idx.numel()) % Ns)              # stream column preserved
        assert (idx[1:] > idx[:-1]).all()                                         # original order
        assert all(want[c] == flag for c in (idx // Ns).unique().tolist())
    # a single odd filter inside a cell drags the whole cell along
    q2 = q.clone(); q2[Ns + 3] = 1e-4
    _, precise2 = B.sweep_partition(q2, r, Ns)
    assert set(range(Ns, 2 * Ns)) <= set(precise2.tolist())
    with pytest.raises(ValueError):
        B.sweep_partition(q[:-1], r[:-1], Ns)


def test_sharded_long_replay_tiles_the_right_columns():
    """Config 5's per-rank input synthesis (workloads.ShardedLongReplay): global filter n follows base trajectory
    n % base_n, so a rank generates exactly columns [begin, end) of the box-wide batch for any window -- on the CPU here
    (same torch code as on the device)."""
    from poseestimationkf_b200 import workloads as W
    N, T, base_n = 5 * 128 * 100 + 640, 12, 1000
    cover = []
    for world in (1, 2, 5):
        for rank in range(world):
            job = W.ShardedLongReplay("cpu", rank=rank, world=world, n_filters=N, n_steps=T, base_n=base_n, chunk_bytes=36 * 7 * N)
            cols = torch.arange(job.begin, job.end) % base_n
            assert job.chunk_steps >= 1 and job.n_local == job.end - job.begin
            for t0, t1 in ((0, min(job.chunk_steps, T)), (T - 1, T)):
                view = job.fill_chunk(t0, t1)
                assert torch.equal(view, job.base.streams[t0:t1][:, :, cols])
            assert torch.equal(job.acc_ref, job.base.acc_ref[:, cols]) and torch.equal(job.mag_ref, job.base.mag_ref[:, cols])
            if world == 5:
                cover.append((job.begin, job.end))
    assert cover[0][0] == 0 and cover[-1][1] == N and all(a[1] == b[0] for a, b in zip(cover, cover[1:]))


def test_bench_workload_selection_and_evidence_stamps():
    """bench.py host logic: the default workload per GPU count (config 2 on one GPU, the sharded config 5 on 2+), the
    executed-arithmetic figures come from the committed opcode census, and the ncu capture whose DRAM traffic the line
    quotes is stamped with the hash of the device sources it was taken from."""
    import argparse
    import json
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    a = argparse.Namespace(workload="auto", filters=None, timesteps=None)
    assert bench.resolve_workload(a, 1) == ("c2", 1 << 20, 1000)
    assert bench.resolve_workload(a, 2) == ("c5", 1 << 24, 2000) and bench.resolve_workload(a, 8)[0] == "c5"
    a.workload, a.filters = "c2", 4096
    assert bench.resolve_workload(a, 8) == ("c2", 4096, 1000)
    assert "configs[4]" in bench.workload_text("c5", 8, 1 << 24, 2000) and "configs[1]" in bench.workload_text("c2", 1, 1 << 20, 1000)
    flops, lane_ops, src = bench.executed_arithmetic("qr2")
    census = json.load(open(os.path.join(root, "profiles", "r02_replay_packed_opcode_census.json")))
    assert flops == census["flops_per_filter_step_executed"] and src.endswith("r02_replay_packed_opcode_census.json")
    assert 200 < lane_ops < 260 and 300 < flops < 400
    sha = bench.kernel_source_sha()
    assert len(sha) == 16 and sha == bench.kernel_source_sha()
    prof = json.load(open(os.path.join(root, "profiles", "r02_replay_packed_ncu_full.json")))
    assert len(prof["kernel_source_sha"]) == 16 and prof["dram_traffic_over_algorithmic"] < 1.1
    assert prof["kernel_source_sha"] == sha, "profiles/r02_replay_packed_ncu_full.json was captured from other device sources: re-profile"
    ref = bench.find_reference()
    assert ref is None or os.path.exists(os.path.join(ref, "ExtendedKalmanFilter.py"))


def test_bench_dump_outputs_and_argument_checks(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy per array; over the byte bound, the same seeded, ordered sample of filter
    columns for every array and for every run.  --steps below 1 and a dump of the reference arm are refused."""
    import bench
    st = B.ReplayState.initial(1000, "cpu", r=0.1)
    st.x = torch.randn(4, 1000, dtype=torch.float64)
    st.loss = torch.arange(1000, dtype=torch.float32)
    arrays = bench.state_arrays(st)
    assert sorted(arrays) == ["state_loss", "state_p", "state_x"]
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, a.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 15 * 4 * 100)          # 15 floats per filter: room for 100 filters
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    keep = np.load(tmp_path / "a" / "state_loss.npy").astype(np.int64)
    assert keep.size == 100 and (np.diff(keep) > 0).all()
    for name, a in arrays.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))
        assert np.array_equal(got, a.float().numpy()[..., keep])
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse()


def test_scale_validation_and_precision_rule_cache():
    """batched._scales_need_precise: validates r > 0, q >= 0 and answers whether any filter needs the precise variant
    (r/q >= 100 or q/r >= 1e4) with one reduction per (q, r) tensor pair; the cached answer must follow in-place writes
    (version counter) and must not survive the tensors themselves (ids are recycled)."""
    q, r = torch.ones(8), torch.full((8,), 0.1)
    assert B._scales_need_precise(q, r) is False and B._scales_need_precise(q, r) is False
    r[3] = 500.0                                    # in-place write: the cached answer is stale
    assert B._scales_need_precise(q, r) is True
    q[5] = 1e5
    r[3] = 0.1
    assert B._scales_need_precise(q, r) is True     # q/r = 1e6 on filter 5
    for _ in range(4):                              # fresh tensors that may reuse the ids / storage of freed ones
        q2, r2 = torch.ones(8), torch.full((8,), 0.1)
        assert B._scales_need_precise(q2, r2) is False
        q3, r3 = torch.ones(8), torch.full((8,), 1000.0)
        assert B._scales_need_precise(q3, r3) is True
        del q2, r2, q3, r3
    for bad_q, bad_r in ((torch.ones(4), torch.zeros(4)), (-torch.ones(4), torch.ones(4)), (torch.ones(4), torch.tensor([1.0, float("nan"), 1.0, 1.0]))):
        with pytest.raises(ValueError):
            B._scales_need_precise(bad_q, bad_r)
    assert B._scales_need_precise(1.0, 0.1) is False and B._scales_need_precise(1e-3, 1e3) is True and B._scales_need_precise(1e3, 1e-3) is True
    with pytest.raises(ValueError):
        B._scales_need_precise(1.0, 0.0)
    assert B._scales_need_precise(2.0, torch.full((4,), 0.5)) is False      # mixed scalar / tensor
