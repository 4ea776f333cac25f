"""CPU: pins the oracle against golden vectors produced by running the REFERENCE'S OWN model code
(tests/golden/make_reference_golden.py: reference classes imported unmodified, executed over an eager
stand-in for the TF-1.x ops -- see tests/golden/tf1_shim.py for what that does and does not prove).

Checked per case (block s=5 / s=8, basis; Toy and a skewed synthetic graph; both sparse_softmax groupings,
i.e. both norm modes of the library): train loss, regularisation, the gradient of every weight, and the
test-mode scores (predict / all subjects / all objects), all in float64 at 1e-10 (norms in float64 too for this
comparison; the oracle's default keeps them as float32 values like the library and TF's float32 op)."""
import os

import numpy as np
import pytest
import torch

from oracle import rgcn_oracle as oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_model_golden.npz")
GOLDEN_TF_KERNEL = os.path.join(os.path.dirname(GOLDEN), "reference_model_golden_tf_kernel.npz")
CASES = [(n, v) for n, v in [("block_toy_s5", "block"), ("block_syn_s8", "block"), ("basis_toy", "basis"),
                             ("basis_syn", "basis")]]
GROUPINGS = [("tf_kernel", "tf_unsorted_compat"), ("canonical", "canonical")]
KEEP = 0.8           # DropoutKeepProbability of both shipped settings files
LAMBDA = 0.01        # RegularizationParameter of both shipped settings files


def _case_arrays(path, name):
    z = np.load(path)
    p = name + "/"
    return {k[len(p):]: z[k] for k in z.files if k.startswith(p)}


def load_case(name):
    """A tf_kernel case is stored as the arrays in which it differs from the canonical case of the same model
    (inputs and weights are shared); tests/golden/make_reference_golden.py writes both files."""
    if name.endswith("_tf_kernel"):
        c = _case_arrays(GOLDEN, name[:-len("tf_kernel")] + "canonical")
        c.update(_case_arrays(GOLDEN_TF_KERNEL, name))
        return c
    return _case_arrays(GOLDEN, name)


# settings file + the overrides the generator applied, per golden case (shared by the CPU-chain and GPU tests)
CASE_SETTINGS = {
    "block_toy_s5": ("gcn_block.exp", {"InternalEncoderDimension": "40", "CodeDimension": "40",
                                       "NumberOfBasisFunctions": "8"}),
    "block_syn_s8": ("gcn_block.exp", {"InternalEncoderDimension": "32", "CodeDimension": "32",
                                       "NumberOfBasisFunctions": "4"}),
    "basis_toy": ("gcn_basis.exp", {"InternalEncoderDimension": "24", "CodeDimension": "24",
                                    "NumberOfBasisFunctions": "5"}),
    "basis_syn": ("gcn_basis.exp", {"InternalEncoderDimension": "20", "CodeDimension": "20",
                                    "NumberOfBasisFunctions": "3"}),
    "basis_toy_1layer": ("gcn_basis.exp", {"InternalEncoderDimension": "24", "CodeDimension": "24",
                                           "NumberOfBasisFunctions": "2", "NumberOfLayers": "1"}),
    "block_toy_1layer": ("gcn_block.exp", {"InternalEncoderDimension": "16", "CodeDimension": "16",
                                           "NumberOfBasisFunctions": "4", "NumberOfLayers": "1"}),
    "distmult_toy": ("distmult.exp", {"CodeDimension": "24"}),
    "block_toy_outproj": ("gcn_block.exp", {"InternalEncoderDimension": "20", "CodeDimension": "12",
                                            "NumberOfBasisFunctions": "4", "UseOutputTransform": "Yes"}),
}


def split_weights(c, variant):
    """Reference get_weights() order (model.py:169-182: next component first): AffineTransform [W, b],
    per layer [W_forward, W_backward, (C_forward, C_backward,) W_self, b], (output AffineTransform [W, b],)
    RelationEmbedding [W_relation].  The graph-less baseline is AffineTransform [W, b] + [W_relation]."""
    n = int(c["n_weights"])
    if variant == "embedding":
        assert n == 3
        return ["W_in", "b_in", "W_relation"], 0
    tail = ["W_out", "b_out", "W_relation"] if variant == "block_outproj" else ["W_relation"]
    variant = "block" if variant == "block_outproj" else variant
    per = 4 if variant == "block" else 6
    n_layers = (n - 2 - len(tail)) // per
    names = ["W_in", "b_in"]
    for l in range(n_layers):
        keys = (["W_forward", "W_backward", "W_self", "b"] if variant == "block"
                else ["W_forward", "W_backward", "C_forward", "C_backward", "W_self", "b"])
        names += ["L%d.%s" % (l, k) for k in keys]
    names += tail
    assert len(names) == n
    return names, n_layers


def oracle_run(c, variant, norm_mode):
    names, n_layers = split_weights(c, variant)
    leaves = {nm: torch.tensor(c["w%d" % i], dtype=torch.float64, requires_grad=True) for i, nm in enumerate(names)}
    p = {"W_in": leaves["W_in"], "b_in": leaves["b_in"],
         "layers": [{k.split(".")[1]: v for k, v in leaves.items() if k.startswith("L%d." % l) and not k.endswith(".b")}
                    for l in range(n_layers)]}
    V, R = int(c["V"]), int(c["R"])
    masks = [c["mask%d" % i] for i in range(int(c["n_masks"]))]

    def encode(graph, mode):
        if variant == "embedding":       # model_builder.py:27-40: codes = W (one-hot input, no bias, no ReLU)
            return oracle.affine_onehot(leaves["W_in"], leaves["b_in"], use_bias=False, use_nonlinearity=False)
        h = oracle.encoder_forward(p, graph, V, R, "block" if variant == "block_outproj" else variant, mode=mode,
                                   drop_masks=masks if mode == "train" else None, keep=KEEP, norm_mode=norm_mode,
                                   dtype=torch.float64, norm_dtype=np.float64)
        if variant == "block_outproj":   # model_builder.py:170-176: linear projection with bias, no ReLU
            h = h @ leaves["W_out"] + leaves["b_out"]
        return h
    codes = encode(c["graph_split"] if variant != "embedding" else None, "train")
    loss, reg, _ = oracle.distmult_loss(codes, leaves["W_relation"], c["X"], c["Y"], torch.float64)
    (loss + LAMBDA * reg).backward()
    with torch.no_grad():
        tc = encode(c["test_graph"], "test").detach()
    return names, leaves, loss.item(), LAMBDA * reg.item(), tc


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-300))


ALL = [(n, v, g, m) for n, v in CASES for g, m in GROUPINGS] + [
    ("basis_toy_1layer", "basis", "canonical", "canonical"), ("block_toy_1layer", "block", "canonical", "canonical"),
    ("distmult_toy", "embedding", "canonical", "canonical"),
    ("block_toy_outproj", "block_outproj", "canonical", "canonical")]


@pytest.mark.parametrize("name,variant,grouping,norm_mode", ALL)
def test_oracle_matches_reference_code_outputs(name, variant, grouping, norm_mode):
    c = load_case(name + "_" + grouping)
    names, leaves, loss, reg, tc = oracle_run(c, variant, norm_mode)
    assert abs(loss - float(c["loss"])) <= 1e-10 * abs(float(c["loss"]))
    assert abs(reg - float(c["reg"])) <= 1e-10 * abs(float(c["reg"]))
    for i, nm in enumerate(names):
        if bool(c["g%d_unused" % i]):
            # only the never-added layer biases (and the baseline's unused input bias) receive no gradient
            assert nm.endswith(".b") or (variant == "embedding" and nm == "b_in"), nm
            assert leaves[nm].grad is None
            continue
        assert rel(leaves[nm].grad.numpy(), c["g%d" % i]) < 1e-10, nm
    Wr, tX = leaves["W_relation"].detach(), c["test_X"]
    e, _ = oracle.distmult_energies(tc, Wr, tX, torch.float64)
    assert rel(torch.sigmoid(e).numpy(), c["predict"]) < 1e-10
    assert rel(oracle.distmult_predict_all_objects(tc, Wr, tX, torch.float64).numpy(), c["all_objects"]) < 1e-10
    assert rel(oracle.distmult_predict_all_subjects(tc, Wr, tX, torch.float64).numpy(), c["all_subjects"]) < 1e-10


def test_golden_is_sensitive_to_the_grouping():
    """The two norm modes genuinely differ on unsorted input (quirk Q1) -- the fixture would catch a mix-up."""
    a, b = load_case("block_toy_s5_tf_kernel"), load_case("block_toy_s5_canonical")
    assert abs(float(a["loss"]) - float(b["loss"])) > 1e-3 * abs(float(b["loss"]))
