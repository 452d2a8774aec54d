"""Host-side pieces of bench.py that need no GPU: the contract of the JSON line depends on them."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_synthetic_ids_survive_the_float32_round_trip_of_the_graph():
    """DIN.py:95,125 feeds the movie ids through float32: the last ids of a 10^8 vocabulary round UP to the
    vocabulary size (TF would assert).  The generator must not draw them - the first cfg-5 sweep of round 2 failed
    on exactly those ids - and must leave small vocabularies alone."""
    from sparrowrecsys_b200.features import synthetic_features
    from sparrowrecsys_b200.spec import baseline_spec
    big = baseline_spec("cfg5_din")
    f = synthetic_features(big, 2048, seed=3, uniform_history=True)
    keys = ["movieId"] + ["userRatedMovie%d" % (k + 1) for k in range(big.hist_len)]
    ids = np.concatenate([np.asarray(f[k]) for k in keys]).astype(np.int64)
    assert ids.max() > 2 ** 26                                    # the whole vocabulary is in play
    assert ids.astype(np.float32).astype(np.int64).max() < big.n_movies
    z = synthetic_features(big, 2048, seed=3)                     # Zipf tail is clipped the same way
    zid = np.concatenate([np.asarray(z[k]) for k in keys]).astype(np.int64)
    assert zid.astype(np.float32).astype(np.int64).max() < big.n_movies
    small = baseline_spec("cfg3_din")
    g = synthetic_features(small, 4096, seed=3, uniform_history=True)
    assert int(np.asarray(g["movieId"]).max()) <= small.n_movies - 1
    assert int(np.asarray(g["movieId"]).max()) > small.n_movies - 200   # ... and still reaches the top of it


def test_tiled_dataset_holds_the_same_rows_in_other_orders():
    import bench
    from sparrowrecsys_b200.features import encode_batch, synthetic_features
    from sparrowrecsys_b200.spec import baseline_spec
    spec = baseline_spec("cfg3_din")
    enc = encode_batch(spec, synthetic_features(spec, 64, seed=5))
    big = bench.tile_encoded(enc, 3, np.random.default_rng(0))
    assert big.B == 3 * 64 and big.hist.shape == (192, enc.hist.shape[1])
    assert np.array_equal(big.hist[:64], enc.hist)                # replica 0 is the original order
    key = lambda e, lo, hi: sorted(map(tuple, np.column_stack([e.movie_id[lo:hi], e.user_id[lo:hi], e.hist[lo:hi]])))
    assert key(big, 64, 128) == key(enc, 0, 64) == key(big, 128, 192)
    assert not np.array_equal(big.hist[64:128], enc.hist)         # ... permuted
    assert bench.tile_encoded(enc, 1, np.random.default_rng(0)) is enc


def test_ncu_traffic_is_only_quoted_for_the_captured_kernel_and_batch():
    import bench
    summary = json.load(open(os.path.join(ROOT, "profiles", "ncu_bench_summary.json")))
    rec = summary["cfg3_din"]
    assert rec["kernel"] == "din_rt_kernel" and rec["batch"] == bench.WORKLOADS["cfg3_din"][0]
    assert bench.ncu_traffic("cfg3_din", "din_rt_kernel", rec["batch"]) == rec["dram_bytes_per_launch"]
    assert bench.ncu_traffic("cfg3_din", "din_rtp_kernel", rec["batch"]) is None    # another kernel
    assert bench.ncu_traffic("cfg3_din", "din_rt_kernel", 2 * rec["batch"]) is None  # another batch size
    assert bench.ncu_traffic("no_such_workload", "din_rt_kernel", 1) is None
    for w, r in summary.items():                                   # every capture is of that workload's own kernel
        assert w in bench.WORKLOADS and r["dram_bytes_per_launch"] > 0 and r["duration_us"] > 0


def test_both_arms_print_the_same_config():
    import bench
    a = bench.parse_args(["--workload", "cfg3_din"])
    b = bench.parse_args(["--workload", "cfg3_din", "--impl", "reference"])
    from sparrowrecsys_b200.spec import baseline_spec
    spec = baseline_spec("cfg3_din")
    assert bench.shared_config(a, spec, 1) == bench.shared_config(b, spec, 1)
    c = bench.shared_config(a, spec, 4)
    assert c["global_batch"] == 4 * c["batch_per_gpu"] and "workload" in c
    assert bench.parse_args(["--workload", "cfg5_din"]).no_graph          # cfg 5 launches directly (DESIGN section 6)
    assert not bench.parse_args(["--workload", "cfg5_din", "--graph"]).no_graph
    assert not bench.parse_args([]).no_graph


def test_stdout_of_the_reference_arm_is_one_json_line():
    """stdout carries the JSON line and nothing else, even when libraries print banners there."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "64",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "inferences/s" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["dtype"] == "f32" and d["higher_is_better"] is True


def test_dumped_outputs_are_bounded_and_the_same_batches_every_run(tmp_path):
    """--dump-outputs: the whole [batches, rows] score array when it fits the limit, otherwise the same seeded
    sample of whole batches on every run, so that two builds can be compared output for output."""
    import pytest
    import torch
    import bench
    scores = torch.arange(64 * 32, dtype=torch.float32).reshape(64, 32)
    bench.dump_outputs(str(tmp_path / "all"), "scores", scores, 1 << 20)
    assert np.array_equal(np.load(tmp_path / "all" / "scores.npy"), scores.numpy())
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), "scores", scores, 10 * 32 * 4)
    a, b = np.load(tmp_path / "a" / "scores.npy"), np.load(tmp_path / "b" / "scores.npy")
    assert a.dtype == np.float32 and a.shape == (10, 32) and np.array_equal(a, b)
    assert len({int(r[0]) // 32 for r in a}) == 10 and all(np.array_equal(r, r[0] + np.arange(32)) for r in a)
    with pytest.raises(SystemExit):
        bench.parse_args(["--impl", "reference", "--dump-outputs", str(tmp_path)])
