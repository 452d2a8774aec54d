"""Candidate retrieval on one GPU: `ItemIndex.search_device` against a torch fp32 baseline in the same run.

Workloads: n in {10^7, 10^8} (both far larger than the 126 MB L2) x dim 64 x q in {1, 16, 128, 256} x
k in {10, 800} x {dot, cosine}, plus one query against the shipped 881 x 10 item2vec catalog (latency).
Time per call = CUDA-event time over a window of >= 200 ms after one warm-up call of the same shape.
Bytes: one scan pass reads n * Dp * 2 bytes (bf16 rows, Dp = round_up(dim, 16) = 64 here) per block of <= 256 queries; the
achieved rate below counts that pass only, so it is a lower bound on the bytes moved when a query needs
extra passes or many survivors are rescored.  The bound is HBM bandwidth (7.7 TB/s data-sheet figure for
a B200 at up to 1,000 W).  Baselines: torch fp32 matmul in row chunks (TF32 off) + torch.topk; for q = 1 and
n <= 10^7 also srs_cosine_scores_device + srs_topk_device (`ranking.rank_by_embedding`'s path).
Prints one JSON line; with --out FILE also writes it there.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return name, power


def timed(fn, min_ms=200.0):
    import torch
    fn()
    torch.cuda.synchronize()
    calls, total = 0, 0.0
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while total < min_ms:
        reps = max(1, calls)
        start.record()
        for _ in range(reps):
            fn()
        end.record()
        end.synchronize()
        total += start.elapsed_time(end)
        calls += reps
    return total / calls


def torch_topk(items, q, k, metric, chunk=1 << 22):
    import torch
    if metric == "cosine":
        q = q / q.norm(dim=1, keepdim=True)
    best_v, best_i = None, None
    for i in range(0, items.shape[0], chunk):
        x = items[i:i + chunk]
        s = q @ x.T
        if metric == "cosine":
            s = s / x.norm(dim=1)[None]
        v, idx = torch.topk(s, min(k, s.shape[1]), dim=1)
        idx = idx + i
        if best_v is None:
            best_v, best_i = v, idx
        else:
            v2, j = torch.topk(torch.cat([best_v, v], 1), k, dim=1)
            best_i = torch.gather(torch.cat([best_i, idx], 1), 1, j)
            best_v = v2
    return best_v, best_i


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="10000000,100000000")
    ap.add_argument("--q", default="1,16,128,256")
    ap.add_argument("--k", default="10,800")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    from sparrowrecsys_b200 import _lib
    from sparrowrecsys_b200.ranking import load_embeddings_csv, rank_by_embedding
    from sparrowrecsys_b200.retrieval import ItemIndex
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures the device and has no CPU fallback")
    torch.backends.cuda.matmul.allow_tf32 = False
    name, power = gpu_info()
    dim = 64
    rows = []
    for n in [int(x) for x in a.n.split(",")]:
        g = torch.Generator(device="cuda").manual_seed(n % 1000)
        items = torch.randn(n, dim, device="cuda", generator=g)
        for metric in ("dot", "cosine"):
            with ItemIndex(items, metric) as ix:
                for nq in [int(x) for x in a.q.split(",")]:
                    q = torch.randn(nq, dim, device="cuda", generator=g)
                    for k in [int(x) for x in a.k.split(",")]:
                        t = timed(lambda: ix.search_device(q, k))
                        tb = timed(lambda: torch_topk(items, q, k, metric))
                        blocks = (nq + 255) // 256
                        Dp = (dim + 15) // 16 * 16                 # the scan copy's padded row width
                        scan_bytes = n * Dp * 2 * blocks
                        row = {"n": n, "dim": dim, "q": nq, "k": k, "metric": metric, "ms": round(t, 4),
                               "torch_fp32_ms": round(tb, 4), "speedup_vs_torch": round(tb / t, 2),
                               "scan_bytes_one_pass": scan_bytes,
                               "achieved_TBps_one_pass": round(scan_bytes / (t * 1e-3) / 1e12, 3),
                               "share_of_hbm_bound": round(scan_bytes / (t * 1e-3) / HBM_BPS, 3)}
                        if nq == 1 and n <= 10 ** 7 and metric == "cosine":
                            qq = q[0].contiguous()
                            scores = torch.empty(n, dtype=torch.float32, device="cuda")
                            lib = _lib.load()

                            def old_path():
                                st = torch.cuda.current_stream().cuda_stream
                                _lib.check(lib.srs_cosine_scores_device(qq.data_ptr(), items.data_ptr(), n, dim,
                                                                        scores.data_ptr(), 0, st))
                                from sparrowrecsys_b200.ranking import topk_device
                                topk_device(scores, k)
                            row["cosine_scores_plus_topk_device_ms"] = round(timed(old_path), 4)
                        rows.append(row)
                        print(json.dumps(row), file=sys.stderr, flush=True)
        del items
        torch.cuda.empty_cache()
    _, M = load_embeddings_csv(os.path.join(ROOT, "tests", "golden", "item2vecEmb.csv"))
    _, U = load_embeddings_csv(os.path.join(ROOT, "tests", "golden", "userEmb_head.csv"))
    with ItemIndex(M, "cosine") as ix:
        Ud = torch.from_numpy(np.ascontiguousarray(U[:1])).cuda()
        lat = timed(lambda: ix.search_device(Ud, 10))
    lat_old = timed(lambda: rank_by_embedding(U[0], M, 10))
    out = {"gpu": name, "power_limit": power, "bound": "HBM bandwidth (scan bytes)", "hbm_TBps_datasheet": 7.7,
           "item2vec_881x10_one_query_ms": round(lat, 4), "rank_by_embedding_881x10_ms": round(lat_old, 4),
           "rows": rows}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
