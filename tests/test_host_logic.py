"""Host-side logic: specs, feature encoding, weight inventory, C-ABI surface."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from sparrowrecsys_b200 import features as F
from sparrowrecsys_b200.spec import (NUMERIC_KEYS, ModelSpec, baseline_spec, default_spec,
                                     history_keys)
from sparrowrecsys_b200.weights import check_weights, init_weights, numeric_rows, weight_shapes


def test_algorithmic_bytes_and_flops_match_survey_8d():
    assert default_spec("embeddingmlp").bytes_per_inference() == 472
    assert default_spec("embeddingmlp").flops_per_inference() == 60416
    assert default_spec("widendeep").bytes_per_inference() == 480
    assert default_spec("widendeep").flops_per_inference() == 60418
    assert default_spec("neuralcf").bytes_per_inference() == 92
    assert default_spec("neuralcf").flops_per_inference() == 620
    assert default_spec("twotowers", hidden=(10,)).flops_per_inference() == 422
    assert baseline_spec("cfg2_deepfm").bytes_per_inference() == 448
    assert baseline_spec("cfg2_deepfm").flops_per_inference() == 13456
    assert baseline_spec("cfg2_deepfm_v2").bytes_per_inference() == 320
    assert baseline_spec("cfg3_din").bytes_per_inference() == 7160
    assert baseline_spec("cfg3_din").flops_per_inference() == 483264
    assert baseline_spec("cfg5_din").bytes_per_inference() == 53072
    assert baseline_spec("cfg5_din").flops_per_inference() == 3466624
    assert default_spec("din").bytes_per_inference() == 428


def test_history_keys_follow_densefeatures_sort():
    assert history_keys(5) == ["userRatedMovie%d" % k for k in range(1, 6)]
    k12 = history_keys(12)
    assert k12[:4] == ["userRatedMovie1", "userRatedMovie10", "userRatedMovie11", "userRatedMovie12"]
    assert k12[4] == "userRatedMovie2"


def test_spec_validation():
    with pytest.raises(ValueError):
        ModelSpec(model="nope")
    with pytest.raises(ValueError):
        default_spec("din", emb_dim=65)
    assert default_spec("din").kind == 6 and default_spec("embeddingmlp").kind == 0


def test_load_samples_csv_semantics(head_rows):
    f = head_rows
    assert f["movieId"].dtype == np.int32 and f["movieAvgRating"].dtype == np.float32
    assert f["movieGenre1"].dtype == object
    # first row of testSamples.csv: userRatedMovie5 is empty -> na_value "0" -> 0
    assert f["userRatedMovie5"][0] == 0 and f["userRatedMovie1"][0] == 349
    assert f["movieGenre1"][0] == "Adventure"
    assert (f["movieGenre3"] == "").sum() > 0            # missing strings stay ""


def test_encode_batch_din(head_rows):
    spec = default_spec("din")
    enc = F.encode_batch(spec, head_rows)
    assert enc.B == 512 and enc.hist.shape == (512, 5) and enc.hist.dtype == np.int32
    assert enc.numerics.shape == (512, 7) and enc.numerics.dtype == np.float32
    np.testing.assert_array_equal(enc.hist[:, 0], head_rows["userRatedMovie1"])
    j = NUMERIC_KEYS.index("releaseYear")
    np.testing.assert_array_equal(enc.numerics[:, j], head_rows["releaseYear"].astype(np.float32))
    assert enc.movie_genre[0, 0] == 2          # "Adventure"
    assert (enc.user_genre[:, 1:] == -1).all()  # DIN reads userGenre1 only
    s = enc.slice(10, 20)
    assert s.B == 10 and s.hist.shape == (10, 5)


def test_encode_batch_errors(head_rows):
    spec = default_spec("neuralcf")
    with pytest.raises(KeyError):
        F.encode_batch(spec, {"movieId": np.array([1])})
    with pytest.raises(ValueError):
        F.encode_batch(spec, {"movieId": np.array([1001]), "userId": np.array([1])})
    with pytest.raises(ValueError):
        F.encode_batch(spec, {"movieId": np.array([1]), "userId": np.array([-3])})
    # unknown keys are ignored, [B,1] columns accepted
    enc = F.encode_batch(spec, {"movieId": np.array([[1], [2]]), "userId": np.array([3, 4]),
                                "rating": np.array([1.0, 2.0])})
    assert enc.B == 2 and enc.hist is None and enc.numerics is None


def test_genre_lookup():
    idx = F.genre_to_index(np.array(["Film-Noir", "Musical", "", "Nope", b"Drama"], dtype=object))
    assert idx.tolist() == [0, 18, -1, -1, 10]
    assert F.genre_to_index(np.array([3, -1])).tolist() == [3, -1]


def test_synthetic_features_shapes():
    spec = baseline_spec("cfg3_din")
    f = F.synthetic_features(spec, 256, seed=2)
    enc = F.encode_batch(spec, f)
    assert enc.hist.shape == (256, 50)
    assert enc.hist.max() < spec.n_movies and enc.hist.min() >= 0
    assert (enc.hist == 0).any()                         # 0-padded tails
    assert (enc.movie_genre[:, 0] == -1).any()           # ~10 % missing genres
    f2 = F.synthetic_features(spec, 256, seed=2)
    assert all(np.array_equal(f[k], f2[k]) for k in f)   # seeded


@pytest.mark.parametrize("model", ["embeddingmlp", "widendeep", "neuralcf", "twotowers",
                                   "deepfm", "deepfm_v2", "din"])
def test_weight_inventory(model):
    spec = default_spec(model)
    W = init_weights(spec, 0)
    check_weights(spec, W)
    names = [n for n, _ in weight_shapes(spec)]
    assert len(names) == len(set(names))
    for k, rows in numeric_rows(spec).items():
        assert len(rows) == 7 and rows.max() < W[k].shape[0]
    bad = dict(W)
    first = names[0]
    bad[first] = np.zeros((3, 3), np.float32)
    with pytest.raises(ValueError):
        check_weights(spec, bad)
    del bad[first]
    with pytest.raises(KeyError):
        check_weights(spec, bad)


def test_din_first_dense_width_matches_reference():
    shapes = dict(weight_shapes(default_spec("din")))
    assert shapes["dense/kernel"] == (57, 128)           # 5E+7 at E=10 (SURVEY.md 8a row a8)
    assert shapes["au_dense/kernel"] == (40, 32) and shapes["au_prelu/alpha"] == (5, 32)
    assert dict(weight_shapes(default_spec("deepfm")))["dense_2/kernel"] == (31040 + 4 + 64, 1)
    assert dict(weight_shapes(default_spec("widendeep")))["dense_2/kernel"] == (10128, 1)


# ---- C ABI --------------------------------------------------------------------------
def _declared_functions():
    with open(os.path.join(ROOT, "include", "srs_ctr.h")) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(srs_[a-z_0-9]+)\s*\(", text)))


def test_abi_library_exports_every_declared_symbol():
    from sparrowrecsys_b200 import _lib
    lib = _lib.load()                      # dlopen only; no CUDA call
    declared = _declared_functions()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(lib, name), "libsrs_ctr.so does not export %s" % name
    assert set(declared) == set(_lib.EXPORTS)
    assert lib.srs_abi_version() == _lib.ABI_VERSION == 3
    assert lib.srs_num_slots() >= 2
    # loading and querying the library launches nothing; checked in a fresh process because the launch counter is
    # per process and GPU tests of the same session may have launched before this one
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); from sparrowrecsys_b200 import _lib; "
                        "lib = _lib.load(); lib.srs_abi_version(); lib.srs_num_slots(); print(lib.srs_launch_count())"
                        % ROOT], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "0", r.stdout + r.stderr


def test_struct_layouts_match_header():
    import ctypes as C
    from sparrowrecsys_b200 import _lib
    assert C.sizeof(_lib.SrsSpec) == 15 * 4
    assert C.sizeof(_lib.SrsTensor) == 40 and _lib.SrsTensor.rows.offset == 16
    assert C.sizeof(_lib.SrsBatch) == 8 + 7 * 8 and _lib.SrsBatch.movie_id.offset == 8
    assert _lib.SrsBatch.hist16.offset == 8 + 6 * 8


def test_product_path_fails_loudly_without_gpu(have_gpu):
    if have_gpu:
        pytest.skip("GPU present")
    from sparrowrecsys_b200 import _lib
    from tfrecmodel import neuralcf
    with pytest.raises(_lib.SrsError) as e:
        neuralcf.load(seed=0)
    assert "no CPU path" in str(e.value)
    with pytest.raises(RuntimeError):
        neuralcf.predict({"movieId": np.array([1]), "userId": np.array([1])})


def test_product_never_imports_oracle():
    bad = []
    for base in ("sparrowrecsys_b200", "tfrecmodel"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            for fn in files:
                if fn.endswith((".py", ".cu", ".cuh", ".h")):
                    with open(os.path.join(dirpath, fn)) as f:
                        src = f.read()
                    if re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M):
                        bad.append(os.path.join(dirpath, fn))
    assert not bad, bad


def test_shard_bounds_cover_rows():
    from sparrowrecsys_b200.sharding import shard_bounds
    for n in (0, 1, 7, 4096, 65536, 65537):
        for w in (1, 2, 3, 8):
            b = [shard_bounds(n, w, r) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1


def test_abi_argument_validation_needs_no_device():
    """Bad arguments are rejected before any CUDA call, with a message (never a fault)."""
    import ctypes as C
    from sparrowrecsys_b200 import _lib
    lib = _lib.load()
    buf = (C.c_float * 4)()
    idx = (C.c_int32 * 4)()
    assert lib.srs_topk_device(buf, -1, 1, idx, None, 0, None) == _lib.SRS_ERR_INVALID
    assert b"negative" in lib.srs_last_error()
    assert lib.srs_topk_device(buf, 4, -2, idx, None, 0, None) == _lib.SRS_ERR_INVALID
    assert lib.srs_topk_device(None, 4, 2, idx, None, 0, None) == _lib.SRS_ERR_INVALID
    assert lib.srs_topk_device(buf, 4, 2, None, None, 0, None) == _lib.SRS_ERR_INVALID
    assert lib.srs_topk_device(None, 0, 5, None, None, 0, None) == _lib.SRS_OK     # nothing to rank
    assert lib.srs_topk_device(buf, 4, 0, None, None, 0, None) == _lib.SRS_OK
    assert lib.srs_rank_host(None, None, 3, idx, buf) == _lib.SRS_ERR_INVALID
    assert lib.srs_predict_host(None, None, buf, None) == _lib.SRS_ERR_INVALID
    assert lib.srs_cosine_scores_device(buf, buf, 4, 0, buf, 0, None) == _lib.SRS_ERR_INVALID
    spec = _lib.SrsSpec()
    spec.kind = 8                                            # one past SRS_DIEN
    h = C.c_void_p()
    assert lib.srs_model_create(C.byref(spec), None, 0, 0, C.byref(h)) == _lib.SRS_ERR_INVALID
    assert b"unknown model kind" in lib.srs_last_error() and not h.value
    with pytest.raises(ValueError):
        default_spec("dien", emb_dim=33)                     # one lane per state element


def test_din_rtp_barrier_protocol_model():
    """din_rtp_kernel (csrc/din_rtp.cu) orders seven roles with nothing but mbarriers across group
    boundaries; its protocol is checked on a CPU model under random interleavings
    (profiles/exp/rtp_protocol_sim.py: no deadlock, no parity aliasing, no operand / staging hazard).
    One-tile groups are the case that deadlocked the first draft."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "rtp_protocol_sim", os.path.join(ROOT, "profiles", "exp", "rtp_protocol_sim.py"))
    sim = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sim)
    for shape in ([1], [14], [14, 14, 14], [1, 1, 1, 1, 1, 1], [2, 1, 3, 1, 1, 2], [16, 1, 5, 16, 1, 1, 7]):
        for seed in range(10):
            sim.Sim(shape, seed).run()


def test_row_tile_barrier_protocol_model():
    """din_rt_kernel / din_rt64_kernel share one mbarrier protocol; profiles/exp/rt_protocol_sim.py runs it on the
    CPU with warp-level actors under random interleavings.  The shipped kernels keep ONE pooling-weights barrier
    per consumer (w_ready[q]); the model shows what that allows when a consumer warp lags its siblings by a tile
    or the issuer is late - a phase completed by arrivals of two different tiles, then parity aliasing and a
    deadlock - and that one barrier per (consumer, pooled buffer) (-DSRS_WREADY_SPLIT, the form din_rtp uses)
    has none of it.  DESIGN.md section 9 item 1."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "rt_protocol_sim", os.path.join(ROOT, "profiles", "exp", "rt_protocol_sim.py"))
    sim = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sim)
    assert sim.check(False, runs=21) == []
    broken = sim.check(True, runs=21)
    assert broken and any("different tiles" in m or "Deadlock" in m or "meant completion" in m for _, _, m in broken)


def test_c_example_builds_against_the_public_header(tmp_path, have_gpu):
    """`include/srs_ctr.h` is a C header (C99, -pedantic clean) and `examples/rank_request.c` - the ranking request
    of RecForYouProcess.java:40-59,113-138 as one call over the C ABI, the body a JNI shim would wrap - compiles,
    links against the library and, without a GPU, fails loudly instead of computing on the CPU."""
    import shutil
    import subprocess
    from sparrowrecsys_b200 import build as B
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    B.build()
    inc = os.path.join(ROOT, "include")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c",
                        os.path.join(inc, "srs_ctr.h")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    exe = str(tmp_path / "rank_request")
    libdir = os.path.dirname(B.LIB)
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", inc,
                        os.path.join(ROOT, "examples", "rank_request.c"), "-L", libdir, "-lsrs_ctr",
                        "-Wl,--unresolved-symbols=ignore-in-shared-libs", "-Wl,-rpath," + libdir, "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    if have_gpu:
        assert run.returncode == 0 and "top 10 of 800 candidates" in run.stdout, run.stdout + run.stderr
    else:
        assert run.returncode == 1 and "no CPU path" in run.stderr
