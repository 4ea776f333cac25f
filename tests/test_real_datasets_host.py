"""CPU: a fixed sample of the real datasets (tests/golden/real_datasets_sample.npz, made by
tests/golden/make_dataset_samples.py) through OUR loaders + host graph preparation, against what the original
project's loader made of the same text (SURVEY.md 8c)."""
import os

import numpy as np
import pytest

from relationprediction_b200.common import io
from relationprediction_b200.ops import Graph
from relationprediction_b200 import _lib

SAMPLE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "real_datasets_sample.npz")


@pytest.mark.parametrize("name", ["FB-Toutanova", "wn18", "FB15k"])
def test_dataset_goldens_and_graph_invariants(toy, tmp_path, name):
    gold = toy["dataset_stats"][name]
    z = np.load(SAMPLE)
    for fname in ("train.txt", "entities.dict", "relations.dict"):
        (tmp_path / fname).write_bytes(z["%s/%s" % (name, fname)].tobytes())
    tr = io.read_triplets_as_array(str(tmp_path / "train.txt"), str(tmp_path / "entities.dict"),
                                   str(tmp_path / "relations.dict"))
    V, R = gold["V"], gold["R"]
    assert (int(z[name + "/V"]), int(z[name + "/R"])) == (V, R)
    np.testing.assert_array_equal(tr, z[name + "/triples"])
    assert tr.dtype == np.int32 and len(tr) > 1000
    g = Graph(tr, V, R)   # host-side build
    info = g.info()
    assert info[0] == 2 * len(tr) and info[3] == 2 * R
    rowptr = g.export(_lib.X_DST_ROWPTR)
    indeg = np.bincount(tr[:, 2], minlength=V) + np.bincount(tr[:, 0], minlength=V)   # fwd into o, bwd into s
    np.testing.assert_array_equal(np.diff(rowptr), indeg)
    norm = g.export(_lib.X_DST_NORM)
    relw = g.export(_lib.X_DST_RELW)
    # per direction the norms of every destination row sum to 1 (or the row has no message of that direction)
    rows = np.repeat(np.arange(V), np.diff(rowptr))
    for lo, hi in ((0, R), (R, 2 * R)):
        sel = (relw >= lo) & (relw < hi)
        sums = np.bincount(rows[sel], weights=norm[sel].astype(np.float64), minlength=V)
        assert np.all((np.abs(sums - 1) < 1e-4) | (sums == 0))
    # (dst, weight id) run count reported by the library == independent count == the count recorded with the sample
    key = rows.astype(np.int64) * (2 * R) + relw
    assert info[9] == 1 + int((key[1:] != key[:-1]).sum()) == int(z[name + "/runs"])
