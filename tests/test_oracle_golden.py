"""Pin the oracle: shipped trained weights of the reference on the bundled test rows
must reproduce the known answers recorded in SURVEY.md section 8c (computed there by
an independent numpy restatement of the graph; TensorFlow itself cannot run here)."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_golden_weights
from oracle import ctr_oracle as O
from sparrowrecsys_b200.spec import default_spec

FIRST8 = [(1, 14887), (10, 11888), (10, 27990), (135, 27108), (15, 23843), (150, 21259),
          (150, 26112), (162, 23843)]
KNOWN = {
    "neuralcf_002": [0.8525178, 0.51808727, 0.35965464, 0.02063905, 0.03719175, 0.80573314,
                     0.5643234, 0.78833336],
    "neuralcf_001": [0.6695241, 0.5660429, 0.08600407, 0.6025467, 0.1260225, 0.9618024,
                     0.59564346, 0.8093899],
    "mlprec_005": [0.5534312, 0.21570465, 0.09113927, 0.37527242, 0.22620608, 0.5138782,
                   0.43187657, 0.9393208],
}


@pytest.fixture(scope="module")
def webroot(tmp_path_factory):
    """The reference's model exports as tests/golden/make_reference_exports.py stored them, unpacked in the layout of
    its `src/main/resources/webroot/modeldata`; returns the directory that holds `modeldata/`."""
    root = tmp_path_factory.mktemp("webroot")
    src = os.path.join(GOLDEN, "modeldata")
    for dirpath, _, files in os.walk(src):
        for name in files:
            dst = root / "modeldata" / os.path.relpath(os.path.join(dirpath, name[:-len(".gz")]), src)
            dst.parent.mkdir(parents=True, exist_ok=True)
            with gzip.open(os.path.join(dirpath, name), "rb") as f:
                dst.write_bytes(f.read())
    return str(root) + os.sep


def test_head_rows_are_the_surveyed_rows(head_rows):
    assert list(zip(head_rows["movieId"][:8].tolist(), head_rows["userId"][:8].tolist())) == FIRST8
    assert len(head_rows["movieId"]) == 512


@pytest.mark.parametrize("name", ["neuralcf_002", "neuralcf_001"])
def test_neuralcf_known_answers(head_rows, name):
    W = load_golden_weights(name)
    sub = {k: v[:8] for k, v in head_rows.items()}
    p, _ = O.neuralcf_forward(default_spec("neuralcf"), W, sub)
    np.testing.assert_allclose(p[:, 0], KNOWN[name], rtol=0, atol=2e-7)
    p64, _ = O.neuralcf_forward(default_spec("neuralcf"), W, sub, dtype=np.float64)
    np.testing.assert_allclose(p64[:, 0], KNOWN[name], rtol=0, atol=2e-7)


def test_twotowers_known_answers(head_rows):
    W = load_golden_weights("mlprec_005")
    sub = {k: v[:8] for k, v in head_rows.items()}
    spec = default_spec("twotowers", hidden=(10,), final_dense=False)
    p, z = O.twotowers_forward(spec, W, sub)
    np.testing.assert_allclose(p[:, 0], KNOWN["mlprec_005"], rtol=0, atol=2e-7)
    assert np.array_equal(p, z)          # raw dot, no sigmoid


def test_httpclient_main_pair():
    """online/util/HttpClient.java:110-147 posts (userId 10351; movieId 52, 53)."""
    W = load_golden_weights("neuralcf_002")
    f = {"movieId": np.array([52, 53], np.int32), "userId": np.array([10351, 10351], np.int32)}
    p, _ = O.neuralcf_forward(default_spec("neuralcf"), W, f)
    np.testing.assert_allclose(p[:, 0], [0.68536943, 0.17321654], rtol=0, atol=2e-7)


def test_full_file_stats_recorded():
    with open(os.path.join(GOLDEN, "full_file_stats.json")) as f:
        s = json.load(f)
    assert s["rows"] == 22440
    assert abs(s["accuracy"] - 0.67879) < 1e-5
    assert abs(s["roc_auc"] - 0.73208) < 1e-5


def test_bundle_reader_matches_fixture(webroot):
    """The TF-free bundle reader on the real SavedModel dirs equals the committed fixture."""
    from sparrowrecsys_b200 import bundle
    W = bundle.load_neuralcf(webroot + "modeldata/neuralcf/002")
    G = load_golden_weights("neuralcf_002")
    for k in ("movieId_embedding", "dense_0/kernel", "dense_0/bias", "dense_1/kernel",
              "dense_2/kernel", "dense_2/bias"):
        assert np.array_equal(W[k], G[k]), k
    nz = np.flatnonzero(np.abs(G["userId_embedding"]).sum(axis=1))
    assert np.array_equal(W["userId_embedding"][nz], G["userId_embedding"][nz])
    idx = bundle.read_index(webroot + "modeldata/neuralcf/002/variables/variables.index")
    e = idx["layer_with_weights-2/kernel/.ATTRIBUTES/VARIABLE_VALUE"]
    assert (e["shape"], e["offset"]) == ((20, 10), 1240080)       # SURVEY.md 8c offsets
    W5 = bundle.load_twotowers(webroot + "modeldata/MLPRec/005")
    assert W5["item_dense_0/kernel"].shape == (10, 10)


def test_head_fixture_is_prefix_of_reference_file():
    """samples_head.csv is byte for byte the start of the reference's testSamples.csv (length and SHA-256 of that
    prefix recorded in reference_files.json)."""
    with open(os.path.join(GOLDEN, "reference_files.json")) as f:
        ref = json.load(f)["sampledata/testSamples.csv"]
    with open(os.path.join(GOLDEN, "samples_head.csv"), "rb") as f:
        head = f.read()
    assert len(head) == ref["prefix_bytes"] and hashlib.sha256(head).hexdigest() == ref["prefix_sha256"]


# ---- the reference's own serialised graphs (tests/golden/make_savedmodel_graph_vectors.py) ----------------
def _graph_vectors():
    with open(os.path.join(GOLDEN, "savedmodel_graph_vectors.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("name", ["neuralcf_002", "neuralcf_001", "mlprec_005"])
def test_oracle_matches_the_serialised_serving_graphs(name):
    """The golden outputs come from evaluating `__inference__wrapped_model_*` of the shipped `saved_model.pb` - the
    function TensorFlow serialised for `serving_default` - node by node (oracle/savedmodel_graph.py), not from a
    reading of the Python scripts: concat order, kernel / bias binding, activations and the Dot tail are the
    graph's.  The oracle must reproduce them on all 512 head rows and the HttpClient pair."""
    v = _graph_vectors()[name]
    W = load_golden_weights(name)
    feats = {"movieId": np.array(v["movieId"], np.int32), "userId": np.array(v["userId"], np.int32)}
    if name == "mlprec_005":
        p, _ = O.twotowers_forward(default_spec("twotowers", hidden=(10,), final_dense=False), W, feats)
    else:
        p, _ = O.neuralcf_forward(default_spec("neuralcf"), W, feats)
    np.testing.assert_allclose(p[:, 0], np.array(v["output"], np.float32), rtol=0, atol=5e-7)
    assert len(v["output"]) == 514
    # the first eight rows are the known answers SURVEY.md 8c recorded, now backed by the graph itself
    np.testing.assert_allclose(v["output"][:8], KNOWN[name], rtol=0, atol=2e-7)


def test_serialised_graph_structure_is_what_the_loaders_assume():
    """Facts read off the graphs that `bundle.load_neuralcf` / `load_twotowers` and the kernels hard-code."""
    v = _graph_vectors()
    for name in ("neuralcf_002", "neuralcf_001"):
        g = v[name]
        assert g["placeholders"] == ["movieId", "userId"]
        assert g["variables"] == {
            "dense_features/movieId_embedding/embedding_weights": "layer_with_weights-0/movieId_embedding/embedding_weights",
            "dense_features_1/userId_embedding/embedding_weights": "layer_with_weights-1/userId_embedding/embedding_weights",
            "dense/kernel": "layer_with_weights-2/kernel", "dense/bias": "layer_with_weights-2/bias",
            "dense_1/kernel": "layer_with_weights-3/kernel", "dense_1/bias": "layer_with_weights-3/bias",
            "dense_2/kernel": "layer_with_weights-4/kernel", "dense_2/bias": "layer_with_weights-4/bias"}
        assert g["dense_features"] == {
            "model/dense_features": ["movieId", "dense_features/movieId_embedding/embedding_weights", 91],
            "model/dense_features_1": ["userId", "dense_features_1/userId_embedding/embedding_weights", 91]}
        w = g["wiring"]
        # movie embedding first, user embedding second into ONE concat (NeuralCF.py:47), then relu, relu, sigmoid
        assert w["model/concatenate/concat"] == ["model/dense_features/concat/concat", "model/dense_features_1/concat/concat",
                                                 "model/concatenate/concat/axis"]
        assert w["model/dense/MatMul"][0] == "model/concatenate/concat" and w["model/dense/Relu"] == ["model/dense/BiasAdd"]
        assert w["model/dense_1/MatMul"][0] == "model/dense/Relu" and w["model/dense_2/MatMul"][0] == "model/dense_1/Relu"
        assert w["model/dense_2/Sigmoid"] == ["model/dense_2/BiasAdd"]
        assert [op for _, op in g["trace"]][-1] == "Identity" and g["trace"][-2] == ["model/dense_2/Sigmoid", "Sigmoid"]
        assert g["nodes_evaluated"] == 196                       # the whole function, sparse lookups and asserts included
    t = v["mlprec_005"]
    w = t["wiring"]
    assert t["variables"]["dense/kernel"] == "layer_with_weights-2/kernel"          # item tower = `dense`
    assert t["dense_features"]["model/dense_features_1"][:2] == ["movieId", "dense_features_1/movieId_embedding/embedding_weights"]
    assert t["dense_features"]["model/dense_features_2"][:2] == ["userId", "dense_features_2/userId_embedding/embedding_weights"]
    assert w["model/dense/MatMul"][0] == "model/dense_features_1/concat/concat"     # one relu Dense per tower
    assert w["model/dense_1/MatMul"][0] == "model/dense_features_2/concat/concat"
    assert w["model/dot/ExpandDims"][0] == "model/dense/Relu" and w["model/dot/ExpandDims_1"][0] == "model/dense_1/Relu"
    assert w["model/dot/Squeeze"] == ["model/dot/MatMul"]
    assert not any(k.endswith("Sigmoid") for k in w)                                # raw Dot(axes=1) output
    assert t["trace"][-2:] == [["model/dot/Squeeze", "Squeeze"], ["Identity", "Identity"]]


def test_feature_column_semantics_read_off_the_older_exports():
    """`modeldata/MLPRec/001-004` are Sequential(DenseFeatures, Dense...) exports over numeric and vocabulary-list
    columns.  No oracle graph corresponds to them, but their serialised functions show the feature-column
    semantics every oracle graph rests on (SURVEY.md 8a): DenseFeatures concatenates its columns sorted by column
    NAME (numeric and categorical interleaved, `<key>_indicator` / `<key>_embedding`), integer numerics are cast to
    float32, a vocabulary list maps word -> list position with -1 for out-of-vocabulary words, "" (strings) and -1
    (ints) mean "no value" and contribute nothing."""
    from sparrowrecsys_b200.spec import GENRE_VOCAB
    v = _graph_vectors()
    for name, width in (("mlprec_001", 6158), ("mlprec_002", 8), ("mlprec_003", 6166), ("mlprec_004", 7)):
        g = v[name]
        assert g["dense_features_order"] == sorted(g["dense_features_order"]), name
        assert g["first_dense_kernel_rows"] == width
    mixed = v["mlprec_003"]["dense_features_order"]
    assert mixed[:6] == ["movieAvgRating", "movieGenre1_indicator", "movieGenre2_indicator", "movieGenre3_indicator",
                         "movieId_indicator", "movieRatingCount"]             # numerics and categoricals interleave
    assert v["mlprec_004"]["dense_features_order"] == ["movieAvgRating", "movieRatingCount", "movieRatingStddev",
                                                       "releaseYear", "userAvgRating", "userRatingCount",
                                                       "userRatingStddev"]    # EmbeddingMLP.py's seven numerics
    assert v["mlprec_004"]["int_columns_cast_to_float"] == ["movieRatingCount", "releaseYear", "userRatingCount"]
    for name in ("mlprec_001", "mlprec_003"):
        g = v[name]
        genres = [c for c in g["vocabularies"] if "genre" in c]
        assert len(genres) == 8
        for c in genres:
            assert g["vocabularies"][c] == list(GENRE_VOCAB), c                 # same words, same order
        assert g["values_are_positions"] and g["oov_default"] == [-1]
        assert all(val == ("" if "Genre" in col else -1) for col, val in g["ignore_value"].items())
        # 8 genre columns x 19 + 6 movie-id columns x 1001 (+ 8 numerics) = the first Dense layer's fan-in
        assert 8 * 19 + 6 * 1001 + (8 if name == "mlprec_003" else 0) == g["first_dense_kernel_rows"]
    # ... and the oracle's conventions are those: position in the list, -1 for unknown / empty words
    f = {"movieGenre1": np.array(["Film-Noir", "Musical", "", "no-such-genre", b"Action"], dtype=object)}
    assert O.genre_index(f, "movieGenre1").tolist() == [0, 18, -1, -1, 1]


def test_identity_column_edge_cases_of_the_serialised_graph(webroot):
    """What the reference's graph itself does with odd ids: an id >= num_buckets trips the graph's own assert (our
    ValueError / SRS_ERR_RANGE), the last valid id works, and -1 is the column's "missing" value: its embedding is
    the zero vector (we reject -1 instead: INTEGRATION.md, error table)."""
    from oracle import savedmodel_graph as SG
    from sparrowrecsys_b200 import bundle
    g = SG.ServingGraph(webroot + "modeldata/neuralcf/002", bundle.read_variables)
    with pytest.raises(ValueError):
        g.run({"movieId": np.array([5, 1001]), "userId": np.array([7, 7])})
    with pytest.raises(ValueError):
        g.run({"movieId": np.array([5, 5]), "userId": np.array([7, 30001])})
    ok = g.run({"movieId": np.array([5, 1000]), "userId": np.array([7, 30000])})
    assert ok.shape == (2, 1)
    W = bundle.load_neuralcf(webroot + "modeldata/neuralcf/002")
    missing = g.run({"movieId": np.array([-1]), "userId": np.array([7])})
    Wz = dict(W)
    Wz["movieId_embedding"] = W["movieId_embedding"].copy()
    Wz["movieId_embedding"][0] = 0                            # row 0 zeroed = what a zero vector does
    p, _ = O.neuralcf_forward(default_spec("neuralcf"), Wz, {"movieId": np.array([0], np.int32), "userId": np.array([7], np.int32)})
    np.testing.assert_allclose(missing[:, 0], p[:, 0], rtol=0, atol=5e-7)
    assert np.array_equal(g.run({"movieId": np.array([3, 9]), "userId": np.array([7, 8])}),
                          g.run({"movieId": np.array([3, 9]), "userId": np.array([7, 8])}, full=False))


def test_graph_vectors_regenerate_from_the_reference_exports(webroot):
    import importlib.util
    spec = importlib.util.spec_from_file_location("mk", os.path.join(GOLDEN, "make_savedmodel_graph_vectors.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    fresh = json.loads(json.dumps(mk.vectors(webroot)))
    assert fresh == _graph_vectors()


def test_whole_test_file_through_the_serialised_graph(webroot):
    """All 22 440 rows of the reference's testSamples.csv through the serialised neuralcf/002 graph
    (full_file_graph.npz): the accuracy / ROC-AUC recorded in full_file_stats.json (SURVEY.md 8c) are the graph's,
    and on the stored sample of rows the graph, evaluated again here, and the oracle agree with it row by row."""
    from oracle import savedmodel_graph as SG
    from sparrowrecsys_b200 import bundle
    z = np.load(os.path.join(GOLDEN, "full_file_graph.npz"))
    pg, lab, rows = z["prob"], z["label"], z["rows"]
    sample = {"movieId": z["movieId"], "userId": z["userId"]}
    g = SG.ServingGraph(webroot + "modeldata/neuralcf/002", bundle.read_variables)
    ps = g.run(sample)[:, 0]
    W = bundle.load_neuralcf(webroot + "modeldata/neuralcf/002")
    po = O.predict(default_spec("neuralcf"), W, sample)[:, 0]
    assert len(pg) == len(lab) == 22440 and len(rows) == 2048
    assert np.abs(ps - pg[rows]).max() <= 5e-7 and np.abs(po - pg[rows]).max() <= 5e-7
    with open(os.path.join(GOLDEN, "full_file_stats.json")) as f:
        s = json.load(f)
    assert abs(float(((pg > 0.5) == (lab == 1)).mean()) - s["accuracy"]) < 1e-9
    order = np.argsort(pg, kind="mergesort")
    ranks = np.empty(len(pg))
    ranks[order] = np.arange(1, len(pg) + 1)
    _, inv, cnt = np.unique(pg, return_inverse=True, return_counts=True)
    ranks = (np.bincount(inv, weights=ranks) / cnt)[inv]
    npos = int((lab == 1).sum())
    auc = (ranks[lab == 1].sum() - npos * (npos + 1) / 2) / (npos * (len(lab) - npos))
    assert abs(auc - s["roc_auc"]) < 1e-6
