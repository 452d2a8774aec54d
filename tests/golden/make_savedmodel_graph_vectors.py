"""Golden vectors from the reference's own serialised graphs:

    python tests/golden/make_savedmodel_graph_vectors.py <SparrowRecSys checkout>

For each shipped export (`modeldata/neuralcf/{002,001}`, `modeldata/MLPRec/005`) `oracle/savedmodel_graph.py`
reads `saved_model.pb`, follows `serving_default` to the `__inference__wrapped_model_*` function TensorFlow wrote,
binds its variables through the export's restore function and evaluates it on the (movieId, userId) pairs of
`samples_head.csv` plus the pair `HttpClient.main` posts (`online/util/HttpClient.java:110-147`).  Written to
`savedmodel_graph_vectors.json`: inputs, outputs, the variable binding and the op trace - what
`tests/test_oracle_golden.py::test_oracle_matches_the_serialised_serving_graphs` holds the oracle to.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import savedmodel_graph as G                               # noqa: E402
from sparrowrecsys_b200 import bundle, features                        # noqa: E402

EXPORTS = {"neuralcf_002": "modeldata/neuralcf/002", "neuralcf_001": "modeldata/neuralcf/001",
           "mlprec_005": "modeldata/MLPRec/005"}


def vectors(webroot):
    """`webroot`: a directory holding the reference's `modeldata/` (its `src/main/resources/webroot`)."""
    rows = features.load_samples_csv(os.path.join(HERE, "samples_head.csv"))
    movie = np.concatenate([np.asarray(rows["movieId"]), [52, 53]]).astype(np.int64)
    user = np.concatenate([np.asarray(rows["userId"]), [10351, 10351]]).astype(np.int64)
    out = {}
    for name, rel in EXPORTS.items():
        g = G.ServingGraph(os.path.join(webroot, rel), bundle.read_variables)
        feeds = {ph: np.zeros(len(movie), np.int64) for ph in g.placeholders.values()}   # unused inputs of MLPRec/005
        feeds["movieId"], feeds["userId"] = movie, user
        y = g.run(feeds).reshape(-1)
        out[name] = {
            "export": rel, "function": g.fn.name, "placeholders": sorted(g.placeholders.values()),
            "variables": {v: k for (v, k) in g.variable_names.values()},
            "dense_features": {k: list(v) for k, v in g.dense_features_blocks().items()},
            "nodes_evaluated": len(g.trace),
            "wiring": {n.name: [i.split(":")[0] for i in n.data_inputs()] for n in g.fn.nodes.values()
                       if "/dense_features" not in n.name and n.op in ("ConcatV2", "MatMul", "BiasAdd", "BatchMatMulV2",
                                                                      "Relu", "Sigmoid", "Squeeze", "ExpandDims")},
            "trace": [[n, op] for n, op in g.trace if "/dense_features" not in n or n.endswith("/concat/concat")],
            "movieId": movie.tolist(), "userId": user.tolist(),
            "output": [float(np.float32(v)) for v in y],
        }
    # the older MLPRec exports are Sequential(DenseFeatures(...), Dense...) models over numeric and vocabulary-list
    # indicator columns: no oracle graph corresponds to them, but they show what DenseFeatures and
    # categorical_column_with_vocabulary_list do - the semantics every other graph of the oracle rests on
    for name, rel in (("mlprec_001", "modeldata/MLPRec/001"), ("mlprec_002", "modeldata/MLPRec/002"),
                      ("mlprec_003", "modeldata/MLPRec/003"), ("mlprec_004", "modeldata/MLPRec/004")):
        g = G.ServingGraph(os.path.join(webroot, rel), bundle.read_variables)
        voc = g.vocabulary_tables()
        casts = sorted(n.name.split("/")[-2] for n in g.fn.nodes.values()
                       if n.op == "Cast" and n.data_inputs()[0] in g.placeholders)
        ignore = {}
        for n in g.fn.nodes.values():
            if n.op == "NotEqual" and "to_sparse_input" in n.name:
                c = g.fn.nodes[n.data_inputs()[1].split(":")[0]]
                v = G.tensor_proto(G.get(c.attr["value"], 8)[0]).reshape(-1)[0]
                ignore[n.name.split("/")[-3]] = v if isinstance(v, str) else int(v)
        out[name] = {
            "export": rel, "function": g.fn.name,
            "dense_features_order": g.dense_features_order(),
            "first_dense_kernel_rows": int(next(v for a, v in g.variables.items() if v.ndim == 2 and "dense_matmul" in a).shape[0]),
            "vocabularies": {c: ([str(k) for k in t["keys"]] if t["keys"].dtype == object else
                                 {"int_keys": int(len(t["keys"])), "keys_are_0_to_n": bool((t["keys"] == np.arange(len(t["keys"]))).all())})
                             for c, t in sorted(voc.items())},
            "values_are_positions": all(bool((t["values"] == np.arange(len(t["values"]))).all()) for t in voc.values()),
            "oov_default": sorted({int(t["default"]) for t in voc.values()}),
            "ignore_value": ignore, "int_columns_cast_to_float": casts,
        }
    return out


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    with open(os.path.join(HERE, "savedmodel_graph_vectors.json"), "w") as f:
        json.dump(vectors(os.path.join(sys.argv[1], "src", "main", "resources", "webroot")), f, indent=0)
    print("wrote savedmodel_graph_vectors.json")
