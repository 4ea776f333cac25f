"""Golden vectors produced by RUNNING THE REFERENCE'S OWN MODEL CODE (needs /root/reference; run HERE):

  python tests/golden/make_reference_golden.py        ->  tests/golden/reference_model_golden.npz
                                                          tests/golden/reference_model_golden_tf_kernel.npz

The reference's model_builder / Representation / AffineTransform / ConcatGcn / BasisGcn / RelationEmbedding /
BilinearDiag classes are imported unmodified from /root/reference/code and executed over tests/golden/tf1_shim.py
(an eager float64 stand-in for the TF-1.x ops they call; TensorFlow 1.4 itself is not installable here).
Settings are the shipped settings/gcn_block.exp and settings/gcn_basis.exp, merged exactly as the reference's
train.py:69-86 does, with only the widths reduced so the fixture stays small.  Weights are drawn by the
reference's own initialisers (numpy RNG, seeded); the decoder batch comes from the reference's NegativeSampler.

Per case the fixture holds: the fed graph and batch, every weight in model.get_weights() order, the dropout
masks in the order the reference drew them (layer 1 then layer 2), and the reference's outputs: train loss,
regularisation, d(loss+reg)/d(weight) for every weight, test-mode sigmoid scores (predict, all subjects,
all objects) with the full training graph fed.  Both sparse_softmax groupings are recorded (see tf1_shim)."""
import os
import sys

import numpy as np
import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(REF, "code"))

import tf1_shim  # noqa: E402
tf = tf1_shim.install()

from common import settings_reader, io, model_builder, auxilliaries, evaluation  # noqa: E402  (reference modules)
from encoders.message_gcns.message_gcn import MessageGcn  # noqa: E402
from decoders.bilinear_diag import BilinearDiag  # noqa: E402


def chain(model):
    while model is not None:
        yield model
        model = model.next_component


def reset_class_level_caches():
    # the reference memoises in CLASS-level dicts (quirk Q5); a fresh process would start from these values
    MessageGcn.vertex_embedding_function = {'train': None, 'test': None}
    BilinearDiag.encoder_cache = {'train': None, 'test': None}


def build(settings_file, overrides, train, V, R, seed):
    settings = settings_reader.read(os.path.join(REF, "settings", settings_file))
    enc, dec, shared, general = settings['Encoder'], settings['Decoder'], settings['Shared'], settings['General']
    for sec, key, val in overrides:
        settings[sec].put(key, val)
    general.put('EntityCount', V)
    general.put('RelationCount', R)
    general.put('EdgeCount', len(train))
    enc.merge(shared)
    enc.merge(general)
    dec.merge(shared)
    dec.merge(general)
    reset_class_level_caches()
    np.random.seed(seed)
    encoder = model_builder.build_encoder(enc, train)
    model = model_builder.build_decoder(encoder, dec)
    model.initialize_train()
    return model, general


class EagerScoringAdapter(object):
    """What Model.score_all_subjects / score_all_objects do through session.run (model.py:59-81), for the eager
    stand-in: feed the registered test graph + the triples, rebuild the test-mode outputs."""

    def __init__(self, model, test_graph):
        self.model, self.test_graph = model, test_graph

    def _feed(self, triplets):
        MessageGcn.vertex_embedding_function['test'] = None
        BilinearDiag.encoder_cache['test'] = None
        for comp in chain(self.model):
            if comp.__class__.__name__ == 'Representation':
                comp.graph = None
        feeds = self.model.get_test_input_variables()
        if self.model.needs_graph():
            feeds[0].feed(self.test_graph)
        feeds[-1].feed(np.asarray(triplets))

    def score_all_subjects(self, triplets):
        self._feed(triplets)
        with torch.no_grad():
            return self.model.predict_all_subject_scores().numpy()

    def score_all_objects(self, triplets):
        self._feed(triplets)
        with torch.no_grad():
            return self.model.predict_all_object_scores().numpy()


def reference_ranking(model, train, ranked):
    """The reference's own Scorer (common/evaluation.py) over the reference model: raw / filtered MRR, Hits@n."""
    sc = evaluation.Scorer({'Metric': 'MRR'})
    sc.register_data(train)
    sc.register_data(ranked)
    sc.register_degrees(train)
    sc.register_model(EagerScoringAdapter(model, train))
    sc.finalize_frequency_computation(np.concatenate((train, ranked), axis=0))
    res = sc.compute_scores(ranked).get_summary().results
    keys = ('MRR', 'H@1', 'H@3', 'H@10')
    return np.array([[float(res[f][k]) for k in keys] for f in ('Raw', 'Filtered')])


def run_case(name, settings_file, overrides, train, test, V, R, seed, grouping, out):
    tf1_shim.SPARSE_SOFTMAX_GROUPING = grouping
    tf1_shim.dropout_rng = np.random.RandomState(seed + 1)
    del tf1_shim.dropout_masks[:]
    model, general = build(settings_file, overrides, train, V, R, seed)
    rng = np.random.RandomState(seed + 2)
    # the per-step sample transform of train.py:201-245, without the neighbourhood sampler
    split = int(float(general['GraphSplitSize']) * len(train))
    graph_split = train[rng.choice(len(train), size=split, replace=False)]
    np.random.seed(seed + 3)
    X, Y = auxilliaries.NegativeSampler(int(general['NegativeSampleRate']), V).transform(train)
    feeds = model.get_train_input_variables()       # [graph_edges, X, Y], or [X, Y] for the graph-less encoder
    if model.needs_graph():
        feeds[0].feed(graph_split)
    feeds[-2].feed(X)
    feeds[-1].feed(Y)
    weights = model.get_weights()
    loss = model.get_loss(mode='train')
    reg = model.get_regularization()
    grads = tf.gradients(loss + reg, weights)
    p = name + "/"
    out[p + "V"], out[p + "R"] = np.int64(V), np.int64(R)
    out[p + "graph_split"] = graph_split.astype(np.int32)
    out[p + "X"], out[p + "Y"] = np.asarray(X, dtype=np.int32), np.asarray(Y, dtype=np.float32)
    out[p + "n_weights"] = np.int64(len(weights))
    for i, (w, g) in enumerate(zip(weights, grads)):
        out[p + "w%d" % i] = w.numpy().astype(np.float32)          # float32-exact: drawn as float32
        out[p + "g%d" % i] = (np.zeros_like(w.numpy()) if g is None else g.numpy())
        out[p + "g%d_unused" % i] = np.bool_(g is None)
    for i, m in enumerate(tf1_shim.dropout_masks):
        out[p + "mask%d" % i] = m
    out[p + "n_masks"] = np.int64(len(tf1_shim.dropout_masks))
    out[p + "loss"], out[p + "reg"] = loss.numpy(), reg.numpy()
    # test mode: full training graph, the reference rebuilds nothing (eager here: drop the frozen graph)
    for comp in chain(model):
        if hasattr(comp, 'graph') and comp.__class__.__name__ == 'Representation':
            comp.graph = None
    tfeeds = model.get_test_input_variables()
    if model.needs_graph():
        tfeeds[0].feed(train)
    tfeeds[-1].feed(test)
    with torch.no_grad():
        out[p + "test_graph"] = train.astype(np.int32)
        out[p + "test_X"] = test.astype(np.int32)
        out[p + "predict"] = model.predict().numpy()
        out[p + "all_subjects"] = model.predict_all_subject_scores().numpy()
        out[p + "all_objects"] = model.predict_all_object_scores().numpy()
    # ranking with the reference's own evaluation code: rows Raw / Filtered, columns MRR, H@1, H@3, H@10
    ranked = np.concatenate((test, train[:40]), axis=0)
    out[p + "ranked"] = ranked.astype(np.int32)
    out[p + "ranking"] = reference_ranking(model, train, ranked)
    print("%-28s loss %.6f reg %.6f  weights %d  masks %d  raw/filtered MRR %.4f %.4f" % (
        name, float(out[p + "loss"]), float(out[p + "reg"]), len(weights), len(tf1_shim.dropout_masks),
        out[p + "ranking"][0, 0], out[p + "ranking"][1, 0]))


def main():
    toy = os.path.join(REF, "data", "Toy")
    ent, rel = os.path.join(toy, "entities.dict"), os.path.join(toy, "relations.dict")
    toy_train = np.array(io.read_triplets_as_list(os.path.join(toy, "train.txt"), ent, rel))
    toy_test = np.array(io.read_triplets_as_list(os.path.join(toy, "test.txt"), ent, rel))
    tV, tR = len(io.read_dictionary(ent)), len(io.read_dictionary(rel))
    rng = np.random.RandomState(11)
    sV, sR, sE = 120, 6, 900
    syn = np.stack([rng.randint(0, sV, sE), rng.randint(0, sR, sE), (rng.zipf(1.6, sE) - 1) % sV], 1)
    syn_test = syn[rng.choice(sE, 12, replace=False)]

    def widths(d, B):
        return [('Encoder', 'InternalEncoderDimension', str(d)), ('Shared', 'CodeDimension', str(d)),
                ('Encoder', 'NumberOfBasisFunctions', str(B))]
    out = {}
    for grouping in ("tf_kernel", "canonical"):
        run_case("block_toy_s5_" + grouping, "gcn_block.exp", widths(40, 8), toy_train, toy_test, tV, tR, 1,
                 grouping, out)
        run_case("block_syn_s8_" + grouping, "gcn_block.exp", widths(32, 4), syn, syn_test, sV, sR, 2,
                 grouping, out)
        run_case("basis_toy_" + grouping, "gcn_basis.exp", widths(24, 5), toy_train, toy_test, tV, tR, 3,
                 grouping, out)
        run_case("basis_syn_" + grouping, "gcn_basis.exp", widths(20, 3), syn, syn_test, sV, sR, 4,
                 grouping, out)
    # BASELINE.json configs[0]: one-layer models (the only layer is also the last one => linear, no ReLU)
    one = [('Encoder', 'NumberOfLayers', '1')]
    run_case("basis_toy_1layer_canonical", "gcn_basis.exp", widths(24, 2) + one, toy_train, toy_test, tV, tR, 5,
             "canonical", out)
    run_case("block_toy_1layer_canonical", "gcn_block.exp", widths(16, 4) + one, toy_train, toy_test, tV, tR, 6,
             "canonical", out)
    # the two remaining factory branches on the path: the graph-less DistMult baseline (settings/distmult.exp,
    # Name=embedding) and the output projection (UseOutputTransform=Yes) on top of the block layers
    run_case("distmult_toy_canonical", "distmult.exp", [('Shared', 'CodeDimension', '24')], toy_train, toy_test,
             tV, tR, 7, "canonical", out)
    run_case("block_toy_outproj_canonical", "gcn_block.exp",
             [('Encoder', 'InternalEncoderDimension', '20'), ('Shared', 'CodeDimension', '12'),
              ('Encoder', 'NumberOfBasisFunctions', '4'), ('Encoder', 'UseOutputTransform', 'Yes')],
             toy_train, toy_test, tV, tR, 8, "canonical", out)
    # a tf_kernel case shares its inputs and weights with the canonical case of the same model: its own file holds
    # only the arrays that differ, which keeps both fixtures under 1 MB (tests/test_reference_golden.py:load_case)
    canonical, tf_kernel = {}, {}
    for k, v in out.items():
        case, arr = k.split("/")
        if not case.endswith("_tf_kernel"):
            canonical[k] = v
            continue
        twin = out[case[:-len("tf_kernel")] + "canonical/" + arr]
        if not (v.dtype == twin.dtype and v.shape == twin.shape and v.tobytes() == twin.tobytes()):
            tf_kernel[k] = v
    np.savez_compressed(os.path.join(HERE, "reference_model_golden.npz"), **canonical)
    np.savez_compressed(os.path.join(HERE, "reference_model_golden_tf_kernel.npz"), **tf_kernel)
    print("wrote reference_model_golden.npz (%d arrays), reference_model_golden_tf_kernel.npz (%d arrays)"
          % (len(canonical), len(tf_kernel)))


if __name__ == "__main__":
    main()
