"""Generates tests/golden/real_datasets_sample.npz from the data/ directory of the original RelationPrediction
checkout:

  python tests/golden/make_dataset_samples.py <RelationPrediction checkout>

Per dataset (FB-Toutanova, wn18, FB15k) the fixture holds a fixed, seeded sample of the real files: the train.txt
lines whose subject AND object fall in a random subset of the entities (file order kept), and the entities.dict /
relations.dict lines of the names those lines use (original ids kept).  Next to the text it stores what the
original project's own loader (common/io.py) makes of it -- the integer triples -- and the number of distinct
(destination, weight id) runs of the graph they form.  tests/test_real_datasets_host.py reads the text with this
project's loader and compares."""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DATASETS = ("FB-Toutanova", "wn18", "FB15k")
TARGET_TRIPLES = 1500


def sample(ref_io, d, seed):
    ent_path, rel_path = os.path.join(d, "entities.dict"), os.path.join(d, "relations.dict")
    ent = ref_io.read_dictionary(ent_path, id_lookup=False)
    with open(os.path.join(d, "train.txt")) as fh:
        lines = fh.read().splitlines(True)
    # an induced subgraph keeps vertices of degree > 1 (a line sample would leave nearly every vertex a leaf)
    keep = np.random.RandomState(seed).random_sample(len(ent)) < (TARGET_TRIPLES / len(lines)) ** 0.5
    rows = [line.rstrip("\n").split("\t") for line in lines]
    train = [line for line, (s, _, o) in zip(lines, rows) if keep[ent[s]] and keep[ent[o]]]
    names = {s for line in train for s in line.rstrip("\n").split("\t")[::2]}
    rels = {line.rstrip("\n").split("\t")[1] for line in train}
    with open(ent_path) as fh:
        ent_lines = [line for line in fh if line.rstrip("\n").split("\t")[1] in names]
    with open(rel_path) as fh:
        rel_lines = [line for line in fh if line.rstrip("\n").split("\t")[1] in rels]
    return "".join(train), "".join(ent_lines), "".join(rel_lines)


def main(checkout):
    sys.path.insert(0, os.path.join(checkout, "code"))
    from common import io as ref_io  # the original project's loader (numpy only)
    out = {}
    for seed, name in enumerate(DATASETS):
        d = os.path.join(checkout, "data", name)
        train, ents, rels = sample(ref_io, d, seed)
        V = len(ref_io.read_dictionary(os.path.join(d, "entities.dict")))
        R = len(ref_io.read_dictionary(os.path.join(d, "relations.dict")))
        with tempfile.TemporaryDirectory() as tmp:
            for fname, text in (("train.txt", train), ("entities.dict", ents), ("relations.dict", rels)):
                with open(os.path.join(tmp, fname), "w") as fh:
                    fh.write(text)
                out["%s/%s" % (name, fname)] = np.frombuffer(text.encode(), np.uint8)
            tr = np.array(ref_io.read_triplets_as_list(os.path.join(tmp, "train.txt"),
                                                      os.path.join(tmp, "entities.dict"),
                                                      os.path.join(tmp, "relations.dict")), dtype=np.int32)
        # one message per direction: forward into the object under r, backward into the subject under R + r
        keys = np.concatenate([tr[:, 2].astype(np.int64) * (2 * R) + tr[:, 1],
                               tr[:, 0].astype(np.int64) * (2 * R) + R + tr[:, 1]])
        out[name + "/triples"] = tr
        out[name + "/V"], out[name + "/R"] = np.int64(V), np.int64(R)
        out[name + "/runs"] = np.int64(len(np.unique(keys)))
        print("%-13s %5d triples, %5d entities, %4d relations, %5d runs" % (
            name, len(tr), ents.count("\n"), rels.count("\n"), int(out[name + "/runs"])))
    np.savez_compressed(os.path.join(HERE, "real_datasets_sample.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
