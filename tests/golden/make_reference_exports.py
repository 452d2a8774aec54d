"""Shrunk copies of the reference's model exports, and what its serialised NeuralCF graph does with its whole
test file, for the tests that hold the oracle to the reference's own graphs:

    python tests/golden/make_reference_exports.py <SparrowRecSys checkout>

Writes, next to this file:

* `modeldata/<export>/<file>.gz` - every file of the exports `neuralcf/{002,001}` and `MLPRec/001-005`,
  gzip-compressed.  `saved_model.pb` and `variables.index` are byte-for-byte.  In `variables.data-*` only the
  float32 model variables of `neuralcf/{002,001}` and `MLPRec/005` are kept, and of their 30001-row user tables
  only the rows the tests use (the users of `samples_head.csv`, of `full_file_graph.npz`, 10351 - the user
  `HttpClient.main` posts - and 7, 8, 30000); every other byte is zero.  `MLPRec/001-004` keep their graphs and
  zeroed variables: the tests read only their structure and the variables' shapes.
* `full_file_graph.npz` - the serialised `neuralcf/002` graph (`oracle/savedmodel_graph.py`) over all 22 440 rows
  of `sampledata/testSamples.csv`: `label` and `prob` for every row, and the `movieId` / `userId` of a seeded
  sample of `rows`, the rows the tests run the graph and the oracle on again.
* `reference_files.json` - length and SHA-256 of the prefix of `testSamples.csv` that `samples_head.csv` copies.
"""
import gzip
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import savedmodel_graph as G                               # noqa: E402
from sparrowrecsys_b200 import bundle, features                        # noqa: E402

EXPORTS = ("neuralcf/002", "neuralcf/001", "MLPRec/001", "MLPRec/002", "MLPRec/003", "MLPRec/004", "MLPRec/005")
WITH_WEIGHTS = ("neuralcf/002", "neuralcf/001", "MLPRec/005")
SAMPLE_ROWS = 2048
EXTRA_USERS = (7, 8, 10351, 30000)


def _model_variable(key, e):
    """The entries `bundle.read_variables` returns (optimizer slots and metric state are not read)."""
    return (e["dtype"] == bundle._DTYPE_FLOAT32 and e["shard"] == 0 and ".OPTIMIZER_SLOT" not in key
            and not key.startswith("optimizer/") and not key.startswith("keras_api/"))


def shrunk_data(variables_dir, users):
    index = bundle.read_index(os.path.join(variables_dir, "variables.index"))
    with open(os.path.join(variables_dir, "variables.data-00000-of-00001"), "rb") as f:
        src = f.read()
    out = bytearray(len(src))
    if users is None:
        return bytes(out)
    for key, e in index.items():
        if not _model_variable(key, e):
            continue
        lo, hi = e["offset"], e["offset"] + e["size"]
        if "userId_embedding" in key:
            row = 4 * e["shape"][1]
            for u in users:
                out[lo + u * row:lo + (u + 1) * row] = src[lo + u * row:lo + (u + 1) * row]
        else:
            out[lo:hi] = src[lo:hi]
    return bytes(out)


def write_gz(path, data):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "wb") as f:                                         # mtime 0: the same bytes on every run
        with gzip.GzipFile(filename="", mode="wb", fileobj=f, mtime=0, compresslevel=9) as g:
            g.write(data)


def main(checkout):
    webroot = os.path.join(checkout, "src", "main", "resources", "webroot")
    test_csv = os.path.join(webroot, "sampledata", "testSamples.csv")
    head_path = os.path.join(HERE, "samples_head.csv")
    with open(head_path, "rb") as f:
        head = f.read()
    with open(test_csv, "rb") as f:
        prefix = f.read(len(head))
    with open(os.path.join(HERE, "reference_files.json"), "w") as f:
        json.dump({"sampledata/testSamples.csv": {"prefix_bytes": len(prefix),
                                                   "prefix_sha256": hashlib.sha256(prefix).hexdigest()}}, f, indent=1)

    full = features.load_samples_csv(test_csv)
    rows = np.sort(np.random.default_rng(2).choice(len(full["userId"]), SAMPLE_ROWS, replace=False))
    g = G.ServingGraph(os.path.join(webroot, "modeldata", "neuralcf", "002"), bundle.read_variables)
    prob = g.run({"movieId": np.asarray(full["movieId"]), "userId": np.asarray(full["userId"])})[:, 0]
    np.savez_compressed(os.path.join(HERE, "full_file_graph.npz"), label=np.asarray(full["label"]).astype(np.int8),
                        prob=prob.astype(np.float32), rows=rows.astype(np.int32),
                        movieId=np.asarray(full["movieId"])[rows].astype(np.int32),
                        userId=np.asarray(full["userId"])[rows].astype(np.int32))

    head_users = set(features.load_samples_csv(head_path)["userId"].tolist()) | set(EXTRA_USERS)
    for rel in EXPORTS:
        src = os.path.join(webroot, "modeldata", rel)
        users = None
        if rel in WITH_WEIGHTS:
            users = head_users | (set(np.asarray(full["userId"])[rows].tolist()) if rel == "neuralcf/002" else set())
            users = sorted(users)
        for dirpath, _, files in os.walk(src):
            for name in files:
                if name.startswith("."):
                    continue
                path = os.path.join(dirpath, name)
                if name.startswith("variables.data"):
                    data = shrunk_data(dirpath, users)
                else:
                    with open(path, "rb") as f:
                        data = f.read()
                write_gz(os.path.join(HERE, "modeldata", rel, os.path.relpath(path, src) + ".gz"), data)
    print("wrote modeldata/, full_file_graph.npz, reference_files.json")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
