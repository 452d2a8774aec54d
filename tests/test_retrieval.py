"""Candidate retrieval (`ItemIndex`, `srs_index_*`): exact top-k dot / cosine search over an item index.

CPU: an fp64 oracle (`retrieve_topk`), checked against the "emb" ranker oracle on the shipped item2vec
embeddings, and a CPU model of the device algorithm (bf16 scan with the margin filter of DESIGN.md
"Candidate retrieval", seed threshold, list capacity, overflow passes, exact fallback) that must agree with
the oracle on adversarial inputs - this is where the margin bound is checked.  GPU: the library against
`rank_by_embedding`, the oracle and float64 torch."""
import math
import os

import numpy as np
import pytest

from oracle import ctr_oracle as O

CAP, SAMPLE, MAX_K = 16384, 16384, 1024          # csrc/retrieve.cu: kCap, kSample, kMaxK


# ---- oracle -----------------------------------------------------------------------------------------------
def rank_keys(s):
    """rank_key() of csrc/rank.cuh: ascending key order = the order of O.rank_topk (descending score, NaN
    first, -0.0 after 0.0, equal scores by lower position)."""
    s = np.asarray(s, np.float32)
    u = s.view(np.uint32).astype(np.uint64)
    mono = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    mono = np.where(np.isnan(s), 0xFFFFFFFF, mono)
    return ((~mono & 0xFFFFFFFF) << np.uint64(32)) | np.arange(len(s), dtype=np.uint64)


def exact_scores(queries, items, metric):
    """fp64 scores [q, n], rounded to float32 (cosine: O.cosine_similarity, Embedding.java:33-47)."""
    q = np.asarray(queries, np.float32).reshape(-1, items.shape[1])
    if metric == "cosine":
        with np.errstate(all="ignore"):
            return np.stack([O.cosine_similarity(v, items) for v in q]).astype(np.float32)
    with np.errstate(all="ignore"):
        return (q.astype(np.float64) @ items.astype(np.float64).T).astype(np.float32)


def retrieve_topk(queries, items, k, metric="dot", exclude=None):
    """Per query the best min(k, eligible) positions by fp64 score in the rank_topk order; unused slots
    position -1, score 0.  Returns (pos int32 [q, k], scores float32 [q, k])."""
    S = exact_scores(queries, items, metric)
    nq, n = S.shape
    pos = np.full((nq, k), -1, np.int32)
    top = np.zeros((nq, k), np.float32)
    for j in range(nq):
        keys = rank_keys(S[j])
        if exclude is not None and exclude[j] >= 0:
            keys[exclude[j]] = np.iinfo(np.uint64).max
        order = np.argsort(keys, kind="stable")
        m = min(k, n - (1 if exclude is not None and exclude[j] >= 0 else 0))
        pos[j, :m] = order[:m]
        top[j, :m] = S[j, order[:m]]
    return pos, top


# ---- CPU model of the device algorithm -----------------------------------------------------------------------
def margin(Dp, metric):
    """csrc/retrieve.cu margin(): bound on |bf16 scan score - exact score| / (|q| |x|)."""
    g = lambda n, u: n * u / (1 - n * u)
    u = 2.0 ** -8
    m = (2 * u + u * u + (1 + u) ** 2 * g(Dp, 2.0 ** -23) + g(Dp, 2.0 ** -24)) * (1 + 2.0 ** -10)
    if metric == "cosine":
        m = m * (1 + 2.0 ** -18) + 2.0 ** -21
    return float(np.nextafter(np.float32(m), np.float32(np.inf)))


def _bf16(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def _scan_operands(a, metric):
    """bf16 scan rows and slack norms as the index / query preparation builds them."""
    a = np.asarray(a, np.float32)
    with np.errstate(all="ignore"):
        if metric == "cosine":
            s = (a * a).astype(np.float64).sum(axis=1)
            bad = ~(s > 0) | ~np.isfinite(s)
            x = (a.astype(np.float64) / np.sqrt(s)[:, None]).astype(np.float32)
            x[bad] = np.nan
            return _bf16(x), np.ones(len(a), np.float32)
        nr = np.sqrt((a.astype(np.float64) ** 2).sum(axis=1)) * (1 + 1e-12)
        nr = nr.astype(np.float32)
        nr = np.where(nr.astype(np.float64) < np.sqrt((a.astype(np.float64) ** 2).sum(axis=1)),
                      np.nextafter(nr, np.float32(np.inf)), nr)
        nr = (nr + np.float32(2.0 ** -50)).astype(np.float32)
        nr[nr >= np.float32(2.0 ** 60)] = np.inf
        return _bf16(a), nr


def model_search(queries, items, k, metric="dot", exclude=None, cap=CAP, sample=SAMPLE, seed=0, stats=None):
    """The device algorithm on the CPU.  The scan score is the fp32 product of bf16-rounded operands; items
    the filter keeps are captured in a random order (the device appends with atomics) up to `cap` entries."""
    import torch
    assert cap > k and sample >= k      # kCap > kMaxK and kSample >= 8 kMaxK on the device
    rng = np.random.default_rng(seed)
    items = np.asarray(items, np.float32)
    q = np.asarray(queries, np.float32).reshape(-1, items.shape[1])
    nq, n = q.shape[0], items.shape[0]
    Dp = (items.shape[1] + 15) // 16 * 16
    m = margin(Dp, metric)
    S = exact_scores(q, items, metric)
    xb, xn = _scan_operands(items, metric)
    qb, qn = _scan_operands(q, metric)
    mq = np.full(nq, m, np.float64) if metric == "cosine" else m * qn.astype(np.float64)
    with np.errstate(all="ignore"):
        approx = (torch.from_numpy(qb) @ torch.from_numpy(xb).T).numpy()          # fp32 accumulation
    PAD = np.iinfo(np.uint64).max
    pos = np.full((nq, k), -1, np.int32)
    top = np.zeros((nq, k), np.float32)
    passes = {"bf16": 0, "exact": 0}
    for j in range(nq):
        ex = -1 if exclude is None else int(exclude[j])
        keys = rank_keys(S[j])
        if ex >= 0:
            keys[ex] = PAD

        def kth(cands):
            kk = np.sort(keys[cands])
            return kk[k - 1] if len(kk) >= k and kk[k - 1] != PAD else PAD

        rng_n = min(n, sample)
        seed_list = np.argsort(keys[:rng_n], kind="stable")[:k]
        seed_list = seed_list[keys[seed_list] != PAD]
        tau = kth(seed_list) if len(seed_list) == k else PAD
        tau_score = -np.inf if tau == PAD else float(S[j, int(tau & 0xFFFFFFFF)])
        final = seed_list
        if n > sample and not (tau != PAD and math.isnan(tau_score)):
            exact, last = False, None
            lst, count = None, 0
            while True:
                if not exact:
                    passes["bf16"] += 1
                    thr = tau_score - mq[j] * xn[sample:].astype(np.float64)
                    with np.errstate(invalid="ignore"):
                        keep = ~(approx[j, sample:] < thr)
                    surv = np.nonzero(keep)[0] + sample
                    surv = surv[surv != ex]
                    cands = np.concatenate([seed_list, rng.permutation(surv)])
                else:
                    passes["exact"] += 1
                    surv = np.nonzero(keys <= tau)[0]
                    cands = rng.permutation(surv)
                count, lst = len(cands), cands[:cap]
                if count <= cap:
                    final = lst
                    break
                if last is not None and count >= last:        # the bf16 scores no longer separate the rows
                    exact = True
                last = count
                new = kth(lst)
                prog = new < tau and not math.isnan(float(S[j, int(new & 0xFFFFFFFF)]))
                tau = new
                tau_score = float(S[j, int(tau & 0xFFFFFFFF)])
                if not prog:                                  # tau did not rise
                    exact = True
        order = np.asarray(final, np.int64)[np.argsort(keys[final], kind="stable")][:k]
        order = order[keys[order] != PAD]
        pos[j, :len(order)] = order
        top[j, :len(order)] = S[j, order]
    if stats is not None:
        stats.update(passes)
    return pos, top


def _assert_same(a, b):
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


# ---- CPU tests ---------------------------------------------------------------------------------------------
def _shipped_embeddings():
    from conftest import GOLDEN
    from sparrowrecsys_b200.ranking import load_embeddings_csv
    mid, M = load_embeddings_csv(os.path.join(GOLDEN, "item2vecEmb.csv"))
    uid, U = load_embeddings_csv(os.path.join(GOLDEN, "userEmb_head.csv"))
    return mid, M, uid, U


EMB_KNOWN = {10292: [875, 15, 424, 433, 387], 19125: [293, 555, 868, 288, 16], 26985: [15, 415, 433, 170, 23]}


def test_oracle_matches_emb_ranker_on_shipped_embeddings():
    mid, M, uid, U = _shipped_embeddings()
    pos, top = retrieve_topk(U, M, 5, "cosine")
    for j in range(len(U)):
        ridx, rtop = O.rank_topk(O.cosine_similarity(U[j], M).astype(np.float32), 5)
        assert np.array_equal(pos[j], ridx) and np.array_equal(top[j], rtop)
        if int(uid[j]) in EMB_KNOWN:
            assert mid[pos[j]].tolist() == EMB_KNOWN[int(uid[j])]
    # similar movies: every movie against the catalog without itself
    ex = np.arange(len(M), dtype=np.int32)
    pos, _ = retrieve_topk(M[:40], M, 10, "cosine", ex[:40])
    for j in range(40):
        s = O.cosine_similarity(M[j], M).astype(np.float32)
        s[j] = -np.inf
        assert j not in pos[j] and np.array_equal(pos[j], O.rank_topk(s, 10)[0])


def test_margin_covers_bf16_error_by_construction():
    """The margin bound against the worst case it is derived for: |q~.x~ - q.x| <= (2u + u^2) sum |q_i x_i|,
    reached when every product rounds the same way."""
    rng = np.random.default_rng(1)
    for Dp in (16, 64, 128):
        m = margin(Dp, "dot")
        assert 2 * 2.0 ** -8 < m < 2 * 2.0 ** -8 * 1.05
        x = rng.uniform(1, 2, (4096, Dp)).astype(np.float32)
        q = rng.uniform(1, 2, Dp).astype(np.float32)
        err = np.abs(_bf16(x).astype(np.float64) @ _bf16(q[None])[0] - x.astype(np.float64) @ q)
        bound = m * np.linalg.norm(q) * np.linalg.norm(x, axis=1)
        assert np.all(err <= bound)


def _adversarial(kind, n, dim, rng):
    if kind == "gaussian":
        return rng.standard_normal((n, dim)).astype(np.float32)
    if kind == "scales":
        return (rng.standard_normal((n, dim)) * 10.0 ** rng.uniform(-3, 3, (n, 1))).astype(np.float32)
    if kind == "near_duplicates":        # differ far below bf16 resolution
        base = rng.standard_normal(dim)
        return (base[None] * (1 + 1e-6 * rng.standard_normal((n, dim)))).astype(np.float32)
    if kind == "cancellation":           # large components that cancel against the query
        a = rng.standard_normal((n, dim)) * 1e3
        a[:, 1::2] = -a[:, 0::2][:, : dim // 2] + rng.standard_normal((n, dim // 2))
        return a.astype(np.float32)
    if kind == "nan_zero":
        a = rng.standard_normal((n, dim)).astype(np.float32)
        a[rng.choice(n, 7, replace=False)] = 0.0
        a[rng.choice(n, 5, replace=False), 0] = np.nan
        return a
    raise ValueError(kind)


def _queries(kind, items, nq, rng):
    dim = items.shape[1]
    if kind == "cancellation":
        return np.ones((nq, dim), np.float32) + 1e-3 * rng.standard_normal((nq, dim)).astype(np.float32)
    return rng.standard_normal((nq, dim)).astype(np.float32)


@pytest.mark.parametrize("metric", ["dot", "cosine"])
@pytest.mark.parametrize("kind", ["gaussian", "scales", "near_duplicates", "cancellation", "nan_zero"])
def test_model_matches_oracle_adversarial(kind, metric):
    rng = np.random.default_rng(len(kind) * 7 + len(metric))
    n, dim = 6000, 24
    items = _adversarial(kind, n, dim, rng)
    q = _queries(kind, items, 4, rng)
    ex = np.array([-1, 3, n - 1, -1], np.int32)
    for k in (1, 50, 300):
        ref = retrieve_topk(q, items, k, metric, ex)
        # a small sample and capacity so that the scan, the overflow passes and the exact path all run
        stats = {}
        _assert_same(model_search(q, items, k, metric, ex, cap=600, sample=1024, stats=stats), ref)
        _assert_same(model_search(q, items, k, metric, ex), ref)
    if kind == "near_duplicates":
        assert stats["exact"] > 0


def test_model_nan_and_zero_rows_rank_first():
    rng = np.random.default_rng(4)
    items = rng.standard_normal((3000, 16)).astype(np.float32)
    items[[5, 2000]] = 0.0
    items[1500, 3] = np.nan
    q = rng.standard_normal((2, 16)).astype(np.float32)
    pos, top = model_search(q, items, 5, "cosine", cap=300, sample=512)
    assert pos[:, :3].tolist() == [[5, 1500, 2000]] * 2 and np.isnan(top[:, :3]).all()
    pos, top = model_search(q, items, 5, "dot", cap=300, sample=512)
    assert pos[:, 0].tolist() == [1500, 1500] and np.isnan(top[:, 0]).all()


def test_model_all_equal_catalog_goes_through_the_overflow_path():
    n, k = 50000, 800
    items = np.ones((n, 8), np.float32)
    q = np.random.default_rng(2).standard_normal((2, 8)).astype(np.float32)
    for metric in ("dot", "cosine"):
        stats = {}
        pos, _ = model_search(q, items, k, metric, stats=stats)
        assert (pos == np.arange(k)).all()
        assert stats["exact"] >= 1


def test_model_k_n_and_exclude_edges():
    rng = np.random.default_rng(8)
    items = rng.standard_normal((700, 12)).astype(np.float32)
    q = rng.standard_normal((3, 12)).astype(np.float32)
    for k in (700, 1000):
        for ex in (None, np.array([0, -1, 699], np.int32)):
            ref = retrieve_topk(q, items, k, "dot", ex)
            _assert_same(model_search(q, items, k, "dot", ex), ref)
            _assert_same(model_search(q, items, min(k, 600), "dot", ex, cap=650, sample=600),
                         retrieve_topk(q, items, min(k, 600), "dot", ex))
    pos, top = retrieve_topk(q, items, 1000, "dot", np.array([0, -1, 699], np.int32))
    assert (pos[0, 699:] == -1).all() and (pos[1, 700:] == -1).all() and (top[0, 699:] == 0).all()
    assert 0 not in pos[0] and 699 not in pos[2]


def test_abi_declares_and_exports_the_retrieval_entry_points():
    import re
    from sparrowrecsys_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "srs_ctr.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    lib = _lib.load()
    for name in ("srs_index_create", "srs_index_destroy", "srs_index_search_device", "srs_index_search_host"):
        assert re.search(r"\b%s\s*\(" % name, text) and name in _lib.EXPORTS and hasattr(lib, name)
    assert "SRS_DOT = 0" in text and "SRS_COSINE = 1" in text
    assert lib.srs_abi_version() == _lib.ABI_VERSION == 3


def test_abi_rejects_bad_index_arguments_without_a_device():
    import ctypes as C
    from sparrowrecsys_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    x = np.zeros((4, 8), np.float32)
    assert lib.srs_index_create(x.ctypes.data, 4, 129, 0, 0, 0, C.byref(h)) == _lib.SRS_ERR_INVALID
    assert lib.srs_index_create(x.ctypes.data, 4, 8, 2, 0, 0, C.byref(h)) == _lib.SRS_ERR_INVALID
    assert lib.srs_index_create(x.ctypes.data, 0, 8, 0, 0, 0, C.byref(h)) == _lib.SRS_ERR_INVALID
    assert lib.srs_index_search_host(None, x.ctypes.data, 1, 8, 5, None, None, None) == _lib.SRS_ERR_INVALID


# ---- GPU tests ---------------------------------------------------------------------------------------------
def _f64_reference(items_t, q, metric, chunk=1 << 20):
    """float64 scores [q, n] on the device, in chunks of rows."""
    import torch
    qd = torch.as_tensor(q, dtype=torch.float64, device=items_t.device)
    if metric == "cosine":
        qd = qd / qd.norm(dim=1, keepdim=True)
    out = []
    for i in range(0, items_t.shape[0], chunk):
        x = items_t[i:i + chunk].double()
        if metric == "cosine":
            x = x / x.norm(dim=1, keepdim=True)
        out.append(qd @ x.T)
    return torch.cat(out, dim=1)


def _check_near_ties(pos, top, ref, k, tol_rel=1e-6):
    """Every position whose fp64 score beats the k-th by more than the tolerance is returned; every returned
    position is within the tolerance of the k-th; returned scores are within 1e-6 relative of fp64."""
    import torch
    for j in range(pos.shape[0]):
        r = ref[j]
        kk = min(k, r.shape[0])
        kth = torch.topk(r, kk).values[-1].item()
        scale = r.abs().max().item()
        tol = 10 * tol_rel * scale + 1e-30
        p = torch.as_tensor(pos[j][pos[j] >= 0].astype(np.int64), device=r.device)
        must = torch.nonzero(r > kth + tol).flatten()
        assert bool(torch.isin(must, p).all()), j
        assert bool((r[p] >= kth - tol).all()), j
        got = torch.as_tensor(top[j][: len(p)].astype(np.float64), device=r.device)
        assert bool(((got - r[p]).abs() <= tol_rel * (r[p].abs() + scale)).all()), j


@pytest.mark.gpu
def test_gpu_shipped_item2vec_matches_rank_by_embedding():
    from sparrowrecsys_b200.ranking import rank_by_embedding
    from sparrowrecsys_b200.retrieval import ItemIndex
    mid, M, uid, U = _shipped_embeddings()
    with ItemIndex(M, "cosine") as ix:
        pos, top = ix.search(U, 5)
    for j in range(len(U)):
        ridx, rtop = rank_by_embedding(U[j], M, 5)
        assert np.array_equal(pos[j], ridx)
        assert np.array_equal(top[j].view(np.uint32), rtop.view(np.uint32))
        if int(uid[j]) in EMB_KNOWN:
            assert mid[pos[j]].tolist() == EMB_KNOWN[int(uid[j])]


@pytest.mark.gpu
def test_gpu_similar_movies_all_881_with_exclude():
    import torch
    from sparrowrecsys_b200.retrieval import ItemIndex
    mid, M, _, _ = _shipped_embeddings()
    ex = np.arange(len(M), dtype=np.int32)
    with ItemIndex(M, "cosine") as ix:
        pos, top = ix.search(M, 20, exclude=ex)                 # 881 queries: four query blocks
        dpos, dtop = ix.search_device(torch.from_numpy(M).cuda(), 20, torch.from_numpy(ex).cuda())
        torch.cuda.synchronize()
    assert np.array_equal(dpos.cpu().numpy(), pos) and np.array_equal(dtop.cpu().numpy(), top)
    assert not (pos == ex[:, None]).any()
    # bit for bit the "emb" ranker's device path (srs_cosine_scores_device + srs_topk_device) with the movie's
    # own score masked
    from sparrowrecsys_b200 import _lib
    from sparrowrecsys_b200.ranking import topk_device
    lib = _lib.load()
    Md = torch.from_numpy(M).cuda()
    scores = torch.empty(len(M), dtype=torch.float32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for j in range(len(M)):
        _lib.check(lib.srs_cosine_scores_device(Md[j].data_ptr(), Md.data_ptr(), len(M), M.shape[1],
                                                scores.data_ptr(), 0, st))
        scores[j] = -float("inf")
        ridx, rtop = topk_device(scores, 20)
        assert np.array_equal(pos[j], ridx.cpu().numpy()), j
        assert np.array_equal(top[j].view(np.uint32), rtop.cpu().numpy().view(np.uint32)), j
    rpos, rtop = retrieve_topk(M, M, 20, "cosine", ex)
    np.testing.assert_allclose(top, rtop, rtol=0, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["dot", "cosine"])
@pytest.mark.parametrize("dim", [10, 16, 64, 128])
def test_gpu_large_synthetic_against_float64(dim, metric):
    import torch
    from sparrowrecsys_b200.retrieval import ItemIndex
    n = 10 ** 6 + 37
    g = torch.Generator(device="cuda").manual_seed(dim)
    items = torch.randn(n, dim, device="cuda", generator=g)
    with ItemIndex(items, metric) as ix:
        for nq in (1, 17, 256, 300):
            q = torch.randn(nq, dim, device="cuda", generator=g)
            ref = _f64_reference(items, q, metric)
            for k in (1, 800, 1024):
                pos, top = ix.search_device(q, k)
                torch.cuda.synchronize()
                pos, top = pos.cpu().numpy(), top.cpu().numpy()
                _check_near_ties(pos, top, ref, k)
                if nq == 17:
                    pos2, top2 = ix.search_device(q, k)
                    assert np.array_equal(pos, pos2.cpu().numpy())
                    assert np.array_equal(top.view(np.uint32), top2.cpu().numpy().view(np.uint32))
    del items


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["dot", "cosine"])
@pytest.mark.parametrize("kind", ["gaussian", "scales", "near_duplicates", "cancellation", "nan_zero"])
def test_gpu_adversarial_against_model_and_oracle(kind, metric):
    from sparrowrecsys_b200.retrieval import ItemIndex
    rng = np.random.default_rng(len(kind) * 13 + len(metric))
    n, dim = 1 << 20, 24
    items = _adversarial(kind, n, dim, rng)
    q = _queries(kind, items, 3, rng)
    ex = np.array([-1, 3, n - 1], np.int32)
    S = exact_scores(q, items, metric)
    with ItemIndex(items, metric) as ix:
        for k in (1, 800):
            pos, top = ix.search(q, k, exclude=ex)
            rpos, rtop = retrieve_topk(q, items, k, metric, ex)
            _assert_same(model_search(q, items, k, metric, ex), (rpos, rtop))   # the CPU model at this size
            for j in range(len(q)):
                s = S[j].astype(np.float64)
                if ex[j] >= 0:
                    s[ex[j]] = -np.inf
                assert ex[j] not in pos[j][pos[j] >= 0]
                nan_ref = np.isnan(rtop[j])
                assert np.array_equal(np.isnan(top[j]), nan_ref) and np.array_equal(pos[j][nan_ref], rpos[j][nan_ref])
                fin = ~nan_ref
                # fp32 rounding of a score is bounded by dim * 2^-24 * sum_i |q_i x_i|, not by the score itself
                with np.errstate(all="ignore"):
                    mag = np.abs(q[j]).astype(np.float64) @ np.abs(items.astype(np.float64)).T
                    if metric == "cosine":
                        mag = mag / (np.linalg.norm(q[j]) * np.linalg.norm(items.astype(np.float64), axis=1))
                tol = 1e-5 * np.nanmax(mag[np.isfinite(mag)]) + 1e-30
                kth = rtop[j][fin][-1].astype(np.float64) if fin.any() else np.inf
                assert np.all(s[pos[j][fin]] >= kth - tol)
                assert np.all(np.abs(top[j][fin].astype(np.float64) - s[pos[j][fin]]) <= tol)


@pytest.mark.gpu
def test_gpu_all_equal_catalog_returns_the_first_positions():
    from sparrowrecsys_b200.retrieval import ItemIndex
    items = np.ones((50000, 8), np.float32)
    q = np.random.default_rng(2).standard_normal((2, 8)).astype(np.float32)
    for metric in ("dot", "cosine"):
        with ItemIndex(items, metric) as ix:
            pos, _ = ix.search(q, 800)
        assert (pos == np.arange(800)).all()


@pytest.mark.gpu
def test_gpu_cfg5_scale_borrowed_table():
    import torch
    from sparrowrecsys_b200 import _lib
    from sparrowrecsys_b200.retrieval import ItemIndex
    n, dim = 10 ** 8, 64
    table = torch.empty(n, dim, dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().srs_fill_uniform(table.data_ptr(), n * dim, 5, -0.05, 0.05, 0,
                                            torch.cuda.current_stream().cuda_stream))
    q = torch.randn(8, dim, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    with ItemIndex(table, "dot") as ix:
        pos, top = ix.search_device(q, 800)
        torch.cuda.synchronize()
    ref = _f64_reference(table, q, "dot", chunk=1 << 24)
    _check_near_ties(pos.cpu().numpy(), top.cpu().numpy(), ref, 800)
    del table, ref


@pytest.mark.gpu
def test_gpu_errors():
    from sparrowrecsys_b200 import _lib
    from sparrowrecsys_b200.retrieval import ItemIndex
    M = np.random.default_rng(0).standard_normal((100, 8)).astype(np.float32)
    with ItemIndex(M, "dot") as ix:
        for k in (0, 1025):
            with pytest.raises(_lib.SrsError) as e:
                ix.search(M[:2], k)
            assert e.value.code == _lib.SRS_ERR_INVALID
        with pytest.raises(_lib.SrsError) as e:
            ix.search(np.zeros((2, 7), np.float32), 5)
        assert e.value.code == _lib.SRS_ERR_INVALID
        for bad in (100, -2):
            with pytest.raises(_lib.SrsError) as e:
                ix.search(M[:2], 5, exclude=np.array([0, bad], np.int32))
            assert e.value.code == _lib.SRS_ERR_INVALID
        pos, _ = ix.search(M[:2], 5, exclude=np.array([0, -1], np.int32))
        assert 0 not in pos[0]
