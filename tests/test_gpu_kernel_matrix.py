"""GPU: one case per compiled instantiation of the aggregation and GEMM kernel templates.

The library picks a template instantiation at run time from d, the block size s = d/B, whether dW is fused into
the backward walk, block_algo and a few RGCN_* knobs.  Every row of CASES names an entry point, a shape, the
algorithm and knobs, and the instantiations the launchers must pick for it (written as in the library, bools as
0/1).  Each case

  * runs under torch.profiler and asserts that every expected kernel appears in the trace;
  * compares every output with a float64 restatement of the same operation, per tensor (max|a-b| / max|b| < 1e-4)
    and ELEMENTWISE (|got - ref| <= C_ELEM * absref, absref = the same float64 computation on |W|, |X|, |norm|),
    so an error confined to a few small elements (one tail slab, one run) cannot hide under the global bar;
  * poisons what must not be read -- NaN weight blocks for unused weight ids, NaN source rows no message reads and
    NaN gradient rows no message reaches -- and checks what must not be written: rows no message targets stay bit
    identical, dW of unused weight ids is exactly 0 (or unchanged bit for bit when accumulating).

The graphs are built so that the weight-id-major work items hit the loop edges: items of 1, GS-1, GS, 31, 32, 33,
64, 65 and item_max messages, runs that cross a group of 8 and an index batch of 32, a run that fills a whole item,
rows 0 and V-1 and rows on both sides of a supertile boundary (RGCN_SUPERTILE_ROWS pinned).  Cases with
RGCN_ITEM_MAX=8 split the destination-major rows, at d > 512 over two column slabs.

tests/test_kernel_matrix_host.py checks on the CPU that CASES (plus a short EXEMPT list) covers every instantiation
in the built library.
"""
import re
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import rgcn_oracle as oracle
from relationprediction_b200 import _lib, ops

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
TOL = 1e-4            # the project's per-tensor bar
# elementwise bar |got - ref| <= C_ELEM * absref.  Worst |got - ref| / absref over all cases: 1.1e-6 (basis-b7-nv3;
# block cases <= 7e-7), NVIDIA B200 at a 1000 W power limit; C_ELEM keeps an 18x margin over it
C_ELEM = 2e-5
ST = 256              # RGCN_SUPERTILE_ROWS pinned for every case
ITEM_MAX = 128        # the library's default work-item length (g.info()[12])


# ---------------------------------------------------------------------------------------------------------------
# kernel names
# ---------------------------------------------------------------------------------------------------------------
_CAST = re.compile(r"\((?:unsigned |signed )?(?:int|bool|char|short|long|long long)\)")


def normalize_kernel_name(name):
    """'void (anonymous namespace)::k_block_team<8, 1, true, true, 4, 4, 3, 8>(const WorkItem *, ...)' (CUPTI) and
    'void <unnamed>::k_block_team<(int)8, (int)1, (bool)1, (bool)1, (int)4, (int)4, (int)3, (int)8>(...)' (cu++filt)
    both become 'k_block_team<8,1,1,1,4,4,3,8>'.  Names without a k_* kernel give None."""
    s = name.replace("(anonymous namespace)::", "").replace("<unnamed>::", "")
    m = re.search(r"\b(k_\w+)", s)
    if not m:
        return None
    base, i = m.group(1), m.end()
    if i >= len(s) or s[i] != "<":
        return base
    depth = 0
    for j in range(i, len(s)):
        if s[j] == "<":
            depth += 1
        elif s[j] == ">":
            depth -= 1
            if depth == 0:
                break
    args = re.sub(r"\s+", "", _CAST.sub("", s[i + 1:j]))
    parts = []
    for a in args.split(","):
        a = {"true": "1", "false": "0"}.get(a, a)
        parts.append(re.sub(r"(?<=\d)[uUlL]+$", "", a))
    return "%s<%s>" % (base, ",".join(parts))


def traced_kernels(fn):
    """Runs fn() under torch.profiler (CUDA activity) and returns (fn's result, set of normalised kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {normalize_kernel_name(e.name) for e in prof.events()}
    names.discard(None)
    return res, names


# ---------------------------------------------------------------------------------------------------------------
# the case table
# ---------------------------------------------------------------------------------------------------------------
Case = namedtuple("Case", "name entry d B algo env expect")
SPLIT = {"RGCN_ITEM_MAX": "8"}


def agg(S, NV):
    return "k_block_agg<%d,%d>" % (S, NV)


def dw(S, NV):
    return "k_block_dw<%d,%d,%d>" % (S, S if S else 4, NV)


def rel(S, NV, F):
    return "k_block_rel<%d,%d,%d>" % (S, NV, F)


def relg(G, F):
    return "k_block_relg<5,%d,%d>" % (G, F)


def stg(S, NV, F, T, NW, NG, GS, MODE):
    return "k_block_stg<%d,%d,%d,%d,%d,%d,%d,%d>" % (S, NV, F, T, NW, NG, GS, MODE)


def team(S, F, T):
    return "k_block_team<%d,1,%d,%d,4,%d,%d,8>" % (S, F, T, 3 if F else 4, 2 if F else 3)


def basis(BC, NV):
    return ["k_basis_agg<%d,%d,0>" % (BC, NV), "k_basis_agg<%d,%d,1>" % (BC, NV), "k_basis_dc<%d,%d>" % (BC, NV)]


STG_FWD_S8 = lambda T: stg(8, 1, 0, T, 16, 3, 8, 1)     # default forward, d > 128
STG_BWD_S8 = lambda T: stg(8, 1, 1, T, 12, 2, 8, 1)     # default fused backward

CASES = [
    # --- block_algo 0: destination-major k_block_agg (forward and dH) + k_block_dw; NV = ceil(d / 128) up to 4
    Case("dst-s4-nv1", "agg", 128, 32, 0, {}, [agg(4, 1), dw(4, 1)]),
    Case("dst-s4-nv2", "layer", 256, 64, 0, {}, [agg(4, 2), dw(4, 2)]),
    Case("dst-s4-nv3", "agg", 384, 96, 0, {}, [agg(4, 3), dw(4, 3)]),
    Case("dst-s4-nv4", "layer", 512, 128, 0, {}, [agg(4, 4), dw(4, 4)]),
    Case("dst-s5-nv1", "layer", 40, 8, 0, {}, [agg(5, 1), dw(5, 1)]),
    Case("dst-s5-nv2", "agg", 200, 40, 0, {}, [agg(5, 2), dw(5, 2)]),
    Case("dst-s5-nv3", "layer", 300, 60, 0, {}, [agg(5, 3), dw(5, 3)]),
    Case("dst-s5-nv4", "agg", 500, 100, 0, {}, [agg(5, 4), dw(5, 4)]),
    Case("dst-s8-nv1", "agg", 64, 8, 0, {}, [agg(8, 1), dw(8, 1)]),
    Case("dst-s8-nv2", "layer", 256, 32, 0, {}, [agg(8, 2), dw(8, 2)]),
    Case("dst-s8-nv3", "agg", 320, 40, 0, {}, [agg(8, 3), dw(8, 2)]),
    Case("dst-s8-nv4", "layer", 512, 64, 0, {}, [agg(8, 4), dw(8, 2)]),
    Case("dst-s16-nv1", "layer", 128, 8, 0, {}, [agg(16, 1), dw(16, 1)]),
    Case("dst-s16-nv2", "agg", 256, 16, 0, {}, [agg(16, 2), dw(16, 1)]),
    Case("dst-s16-nv3", "layer", 384, 24, 0, {}, [agg(16, 3), dw(16, 1)]),
    Case("dst-s16-nv4", "agg", 512, 32, 0, {}, [agg(16, 4), dw(16, 1)]),
    Case("dst-s6-nv1", "agg", 24, 4, 0, {}, [agg(0, 1), dw(0, 1)]),
    Case("dst-s6-nv2", "layer", 240, 40, 0, {}, [agg(0, 2), dw(0, 2)]),
    Case("dst-s6-nv3", "agg", 360, 60, 0, {}, [agg(0, 3), dw(0, 3)]),
    Case("dst-s6-nv4", "layer", 480, 80, 0, {}, [agg(0, 4), dw(0, 4)]),
    # split rows (several warp items per row, last-arriver epilogue) with two column slabs, one counter per slab
    Case("dst-s8-d1024-split", "agg", 1024, 128, 0, SPLIT, [agg(8, 4), dw(8, 2)]),
    Case("dst-s4-d640-split", "layer", 640, 160, 0, SPLIT, [agg(4, 4), dw(4, 4)]),
    Case("dst-s2-d768-split", "agg", 768, 384, 0, SPLIT, [agg(0, 4), dw(0, 4)]),
    Case("dst-s5-split", "layer", 500, 100, 0, SPLIT, [agg(5, 4), dw(5, 4)]),
    # --- block_algo 1: weight-id-major, rows in registers; the dW-fused backward runs with one quad per lane
    Case("rel-s4-nv1", "agg", 128, 32, 1, {}, [rel(4, 1, 0), rel(4, 1, 1)]),
    Case("rel-s4-nv2", "layer", 256, 64, 1, {}, [rel(4, 2, 0), rel(4, 1, 1)]),
    Case("rel-s4-nv3", "agg", 384, 96, 1, {}, [rel(4, 3, 0), rel(4, 1, 1)]),
    Case("rel-s4-nv4", "layer", 512, 128, 1, {}, [rel(4, 4, 0), rel(4, 1, 1)]),
    Case("rel-s8-nv1", "layer", 128, 16, 1, {}, [rel(8, 1, 0), rel(8, 1, 1)]),
    Case("rel-s8-nv2", "agg", 512, 64, 1, {}, [rel(8, 2, 0), rel(8, 1, 1)]),
    Case("rel-s8-d1024", "agg", 1024, 128, 1, {}, [rel(8, 2, 0), rel(8, 1, 1)]),
    Case("rel-s16", "layer", 256, 16, 1, {}, [rel(16, 1, 0), rel(16, 1, 1)]),
    Case("relg-g4", "layer", 500, 100, 1, {}, [relg(4, 0), relg(4, 1)]),
    Case("relg-g2", "agg", 200, 40, 1, {"RGCN_REL_GROUP": "2"}, [relg(2, 0), relg(2, 1)]),
    # one-warp s = 5 kernel (RGCN_REL_GROUP outside {2, 4}): dH by k_block_rel, dW by k_block_dw
    Case("rel-s5-nv1", "agg", 40, 8, 1, {"RGCN_REL_GROUP": "1"}, [rel(5, 1, 0), dw(5, 1)]),
    Case("rel-s5-nv2", "layer", 200, 40, 1, {"RGCN_REL_GROUP": "1"}, [rel(5, 2, 0), dw(5, 2)]),
    Case("rel-s5-nv3", "agg", 300, 60, 1, {"RGCN_REL_GROUP": "1"}, [rel(5, 3, 0), dw(5, 3)]),
    Case("rel-s5-nv4", "layer", 500, 100, 1, {"RGCN_REL_GROUP": "1"}, [rel(5, 4, 0), dw(5, 4)]),
    # --- block_algo 3: TMA / cp.async staged weight-id-major kernels; TAIL = the last slab is narrower
    Case("stg-s4", "agg", 256, 64, 3, {}, [stg(4, 1, 0, 0, 16, 3, 8, 1), stg(4, 1, 1, 0, 12, 2, 8, 1)]),
    Case("stg-s4-tail", "layer", 260, 65, 3, {}, [stg(4, 1, 0, 1, 16, 3, 8, 1), stg(4, 1, 1, 1, 12, 2, 8, 1)]),
    Case("stg-s8-d64", "layer", 64, 8, 3, {}, [stg(8, 1, 0, 1, 16, 3, 8, 0), STG_BWD_S8(1)]),
    Case("stg-s8-d128", "agg", 128, 16, 3, {}, [stg(8, 1, 0, 0, 16, 3, 8, 0), STG_BWD_S8(0)]),
    Case("stg-s8", "layer", 256, 32, 3, {}, [STG_FWD_S8(0), STG_BWD_S8(0)]),
    Case("stg-s8-tail", "agg", 264, 33, 3, {}, [STG_FWD_S8(1), STG_BWD_S8(1)]),
    Case("stg-s8-d1024", "agg", 1024, 128, 3, {}, [STG_FWD_S8(0), STG_BWD_S8(0)]),
    Case("stg-s8-nv2", "agg", 256, 32, 3, {"RGCN_STG_FWD": "0", "RGCN_STG_BWD": "3"},
         [stg(8, 2, 0, 0, 12, 2, 8, 0), stg(8, 2, 1, 0, 8, 2, 4, 0)]),
    Case("stg-s8-nv2-tail", "layer", 264, 33, 3, {"RGCN_STG_FWD": "0", "RGCN_STG_BWD": "3"},
         [stg(8, 2, 0, 1, 12, 2, 8, 0), stg(8, 2, 1, 1, 8, 2, 4, 0)]),
    Case("stg-s8-tma", "layer", 256, 32, 3, {"RGCN_STG_FWD": "2", "RGCN_STG_BWD": "0"},
         [stg(8, 1, 0, 0, 16, 3, 8, 0), stg(8, 1, 1, 0, 12, 2, 8, 0)]),
    Case("stg-s8-tma-tail", "agg", 264, 33, 3, {"RGCN_STG_FWD": "2", "RGCN_STG_BWD": "0"},
         [stg(8, 1, 0, 1, 16, 3, 8, 0), stg(8, 1, 1, 1, 12, 2, 8, 0)]),
    Case("stg-s16", "agg", 256, 16, 3, {}, [stg(16, 1, 0, 0, 16, 3, 8, 1), stg(16, 1, 1, 0, 8, 2, 8, 1)]),
    Case("stg-s16-tail", "layer", 144, 9, 3, {}, [stg(16, 1, 0, 1, 16, 3, 8, 1), stg(16, 1, 1, 1, 8, 2, 8, 1)]),
    # team kernels (384 < d <= 512, s in {4, 8}); d % 128 != 0 gives the TAIL variants
    Case("team-s8", "layer", 512, 64, 3, {}, [team(8, 0, 0), team(8, 1, 0)]),
    Case("team-s8-tail", "agg", 400, 50, 3, {}, [team(8, 0, 1), team(8, 1, 1)]),
    Case("team-s4", "agg", 512, 128, 3, {}, [team(4, 0, 0), team(4, 1, 0)]),
    Case("team-s4-tail", "layer", 500, 125, 3, {}, [team(4, 0, 1), team(4, 1, 1)]),
    Case("team-s8-tail-auto", "layer", 400, 50, -1, {}, [team(8, 0, 1), team(8, 1, 1)]),
    # --- basis layer: (bases per pass BC, NV) for the forward (layout 0), dH (layout 1) and dC kernels
    Case("basis-b1-nv1", "basis", 128, 1, -1, {}, basis(1, 1)),
    Case("basis-b1-nv2", "basis", 256, 1, -1, {}, basis(1, 2)),
    Case("basis-b1-nv3", "basis", 384, 1, -1, {}, basis(1, 3)),
    Case("basis-b1-nv4", "basis", 512, 1, -1, {}, basis(1, 4)),
    Case("basis-b2-nv1", "basis", 64, 2, -1, {}, basis(2, 1)),
    Case("basis-b2-nv2", "basis", 200, 2, -1, {}, basis(2, 2)),
    Case("basis-b2-nv3", "basis", 300, 2, -1, {}, basis(2, 3)),
    Case("basis-b2-nv4", "basis", 500, 2, -1, {}, basis(2, 4)),
    Case("basis-b3-nv1", "basis", 96, 3, -1, {}, basis(4, 1)),
    Case("basis-b4-nv2", "basis", 240, 4, -1, {}, basis(4, 2)),
    Case("basis-b7-nv3", "basis", 360, 7, -1, {}, basis(4, 3)),
    Case("basis-b4-nv4", "basis", 480, 4, -1, {}, basis(4, 4)),
    Case("basis-b5-nv1", "basis", 40, 5, -1, {}, basis(5, 1)),
    Case("basis-b5-nv2", "basis", 200, 5, -1, {}, basis(5, 2)),
    Case("basis-b5-nv3", "basis", 300, 5, -1, {}, basis(5, 3)),
    Case("basis-b5-nv4", "basis", 500, 5, -1, {}, basis(5, 4)),
    Case("basis-b2-d640-split", "basis", 640, 2, -1, SPLIT, basis(2, 4)),
    Case("basis-b5-split", "basis", 300, 5, -1, SPLIT, basis(5, 3)),
    # --- GEMMs
    Case("gemm-nt", "gemm", 0, 0, -1, {}, ["k_split_b", "k_gemm_tf32x3<0>"]),
    Case("gemm-rank", "rank", 0, 0, -1, {}, ["k_gemm_tf32x3<1>"]),
    Case("gemm-tn", "tn", 0, 0, -1, {}, ["k_gemm_tn_tf32x3<3>"]),
]

# instantiations that are in the library but have no row above, with the reason
EXEMPT = {
    "k_gemm_tn_tf32x3<2>": "RGCN_GEMM_PF=2 is read once per process: test_gpu_gemm.py runs it in a child process "
                           "and checks the kernel name there",
}


# ---------------------------------------------------------------------------------------------------------------
# graphs with loop edges
# ---------------------------------------------------------------------------------------------------------------
def item_lengths(item_max):
    return [1, 3, 4, 7, 8, 9, 31, 32, 33, 64, 65, item_max, item_max + 37]


PATTERNS = ("one", "nine", "cross", "distinct", "mixed")


def run_lengths(L, pattern, rng):
    """Multiplicities of consecutive rows in one (supertile, weight id) segment of L messages."""
    if pattern == "one":                    # one run fills the whole item
        return [L]
    if pattern == "nine":                   # runs of 9 cross every group of 8
        return [9] * (L // 9) + ([L % 9] if L % 9 else [])
    if pattern == "cross":                  # runs over messages 28..36 and 60..68: across index batches of 32
        cuts = [c for c in (28, 37, 60, 69) if c < L]
        edges = [0] + cuts + [L]
        return [b - a for a, b in zip(edges[:-1], edges[1:])]
    if pattern == "distinct":
        return [1] * L
    out = []
    while sum(out) < L:
        out.append(min(int(rng.randint(1, 6)), L - sum(out)))
    return out


def segment_rows(n_rows, t, runs, quiet, rng):
    """Distinct rows of supertile t, one per run, ascending; the supertile's edge rows (0, V-1, both sides of the
    boundaries) come first."""
    lo, hi = t * ST, min((t + 1) * ST, n_rows)
    special = [r for r in (lo, lo + ST - 1, n_rows - 1) if lo <= r < hi and r not in quiet]
    pool = np.setdiff1d(np.arange(lo, hi), np.concatenate([quiet, special]))
    k = len(runs)
    take = special[:k]
    take = take + list(rng.choice(pool, k - len(take), replace=False))
    rows = np.sort(np.array(take, dtype=np.int64))
    return np.repeat(rows, runs)


def designed_pairs(n_a, n_b, n_w, unused, quiet_a, quiet_b, item_max, rng):
    """Messages (a, b, w) over weight ids w: for even w the a side follows the loop-edge design (segment lengths
    and runs per a-supertile), for odd w the b side; the other side is random over its non-quiet rows."""
    lengths = item_lengths(item_max)
    A, Bs, W = [], [], []
    k = 0
    for w in range(n_w):
        if w in unused:
            continue
        des_n, des_q, oth_n, oth_q = (n_a, quiet_a, n_b, quiet_b) if w % 2 == 0 else (n_b, quiet_b, n_a, quiet_a)
        oth_pool = np.setdiff1d(np.arange(oth_n), oth_q)
        for t in range((des_n + ST - 1) // ST):
            L = lengths[k % len(lengths)]
            pat = PATTERNS[(k + k // len(lengths)) % len(PATTERNS)]
            k += 1
            rows = segment_rows(des_n, t, run_lengths(L, pat, rng), des_q, rng)
            other = rng.choice(oth_pool, len(rows))
            a, b = (rows, other) if w % 2 == 0 else (other, rows)
            A.append(a)
            Bs.append(b)
            W.append(np.full(len(rows), w))
    return (np.concatenate(A).astype(np.int32), np.concatenate(Bs).astype(np.int32),
            np.concatenate(W).astype(np.int32))


# ---------------------------------------------------------------------------------------------------------------
# checks
# ---------------------------------------------------------------------------------------------------------------
WORST = {}


def np64(x):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu()
        return x.numpy().astype(np.float64)
    return np.asarray(x, dtype=np.float64)


def check(case, name, got, ref, absref):
    got, ref, absref = np64(got), np64(ref), np64(absref)
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert np.isfinite(got).all(), "%s: %s has non-finite values" % (case.name, name)
    e = float(np.abs(got - ref).max() / (np.abs(ref).max() + 1e-30))
    assert e < TOL, "%s: %s rel err %.3e >= %.1e" % (case.name, name, e, TOL)
    diff = np.abs(got - ref)
    bad = diff > C_ELEM * absref
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(absref > 0, diff / absref, np.where(diff > 0, np.inf, 0.0))
    worst = float(ratio.max()) if ratio.size else 0.0
    WORST[(case.name, name)] = worst
    if bad.any():
        idx = np.argwhere(bad)[:5].tolist()
        raise AssertionError("%s: %s fails the elementwise bar at %d elements (first %s), worst |err|/absref %.3e"
                             % (case.name, name, int(bad.sum()), idx, worst))


def block_weights(rng, n_w, B, s, unused):
    """(reference weights with zero blocks for the unused weight ids, kernel weights with NaN blocks there)"""
    W = rng.normal(0, 0.3, (n_w, B, s, s)).astype(np.float32)
    W[list(unused)] = 0
    Wk = W.copy()
    Wk[list(unused)] = np.nan
    return W, Wk


# ---------------------------------------------------------------------------------------------------------------
# entry points
# ---------------------------------------------------------------------------------------------------------------
def run_agg(case, item_max):
    """rgcn_block_aggregate / _backward over a messages-only graph with separate source rows (V_src > V_dst)."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    d, B = case.d, case.B
    s = d // B
    V_dst, V_src, n_w = 3 * ST - 60, 4 * ST - 30, 12
    unused = {3, 10}
    quiet_dst = rng.choice(np.setdiff1d(np.arange(V_dst), [0, ST - 1, ST, 2 * ST - 1, 2 * ST, V_dst - 1]), 40, False)
    quiet_src = rng.choice(np.setdiff1d(np.arange(V_src), np.arange(0, V_src, ST).tolist()
                                        + np.arange(ST - 1, V_src, ST).tolist() + [V_src - 1]), 60, False)
    dst, src, relw = designed_pairs(V_dst, V_src, n_w, unused, quiet_dst, quiet_src, item_max, rng)
    M = len(dst)
    norm = rng.uniform(0.1, 1.0, M).astype(np.float32)
    g = ops.Graph.from_messages(dst, src, relw, norm, V_dst, V_src, n_w, device=0)
    assert g.info()[12] == item_max
    W, Wk = block_weights(rng, n_w, B, s, unused)
    R = n_w // 2
    X = rng.normal(0, 1, (V_src, d)).astype(np.float32)
    G = rng.normal(0, 1, (V_dst, d)).astype(np.float32)
    read = np.zeros(V_src, bool)
    read[src] = True
    reached = np.zeros(V_dst, bool)
    reached[dst] = True
    assert (~read).sum() >= 60 and (~reached).sum() >= 40
    Xk, Gk = X.copy(), G.copy()
    Xk[~read] = np.nan
    Gk[~reached] = np.nan
    out0 = rng.normal(0, 1, (V_dst, d)).astype(np.float32)
    dW0 = rng.normal(0, 1, (n_w, B, s, s)).astype(np.float32)

    cu = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    Xt, Gt, Wft, Wbt = cu(Xk), cu(Gk), cu(Wk[:R]), cu(Wk[R:])

    def fn():
        out = cu(out0)
        ops.block_aggregate_(out, Xt, Wft, Wbt, g, B)
        dX, dWf, dWb = ops.block_aggregate_backward(Xt, Wft, Wbt, Gt, g, B)
        aWf, aWb = cu(dW0[:R]), cu(dW0[R:])
        ops.block_aggregate_backward(Xt, Wft, Wbt, Gt, g, B, aWf, aWb)
        return out, dX, torch.cat([dWf, dWb]), torch.cat([aWf, aWb])

    (out, dX, dWk, adW), names = traced_kernels(fn)

    # float64 restatement: out[dst] += norm W[relw] . X[src] per block; autograd for dX and dW
    def ref(Xv, Wv, nv, Gv):
        Xr = torch.tensor(Xv, dtype=torch.float64, requires_grad=True)
        Wr = torch.tensor(Wv, dtype=torch.float64, requires_grad=True)
        idx = lambda a: torch.as_tensor(a.astype(np.int64))
        msg = torch.einsum("mbij,mbj->mbi", Wr[idx(relw)], Xr[idx(src)].reshape(M, B, s))
        msg = msg.reshape(M, d) * torch.tensor(nv, dtype=torch.float64)[:, None]
        o = torch.zeros(V_dst, d, dtype=torch.float64).index_add(0, idx(dst), msg)
        o.backward(torch.tensor(Gv, dtype=torch.float64))
        return o.detach().numpy(), Xr.grad.numpy(), Wr.grad.numpy()

    r_out, r_dX, r_dW = ref(X, W, norm, G)
    a_out, a_dX, a_dW = ref(np.abs(X), np.abs(W), np.abs(norm), np.abs(G))
    check(case, "out", out, out0 + r_out, np.abs(out0) + a_out)
    check(case, "dX", dX, r_dX, a_dX)
    check(case, "dW", dWk, r_dW, a_dW)
    check(case, "dW accumulated", adW, dW0 + r_dW, np.abs(dW0) + a_dW)
    out, dX, dWk, adW = (t.cpu().numpy() for t in (out, dX, dWk, adW))
    assert np.array_equal(out[~reached].view(np.int32), out0[~reached].view(np.int32)), "untargeted rows changed"
    assert (dX[~read] == 0).all(), "dX of unread source rows"
    assert (dWk[list(unused)] == 0).all(), "dW of unused weight ids"
    assert np.array_equal(adW[list(unused)].view(np.int32), dW0[list(unused)].view(np.int32)), \
        "accumulated dW of unused weight ids changed"
    return names


def layer_graph(rng, V, R, unused_rel, item_max):
    o, s_, r = designed_pairs(V, V, R, {unused_rel}, np.zeros(0, np.int64), np.zeros(0, np.int64), item_max, rng)
    tr = np.stack([s_, r, o], 1).astype(np.int32)
    nf = rng.uniform(0.1, 1.0, len(tr)).astype(np.float32)
    nb = rng.uniform(0.1, 1.0, len(tr)).astype(np.float32)
    g = ops.Graph(tr, V, R, norm_mode="explicit", norm_f=nf, norm_b=nb, device=0)
    assert g.info()[12] == item_max
    return tr, nf, nb, g


def run_layer(case, item_max):
    """block_layer forward + backward against oracle.layer_fwd_bwd (no ReLU: the elementwise bar needs a linear
    layer; the ReLU / dropout epilogues are covered by test_gpu_parity.py)."""
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    d, B = case.d, case.B
    s = d // B
    V, R, unused = 3 * ST - 40, 6, 4
    tr, nf, nb, g = layer_graph(rng, V, R, unused, item_max)
    H = rng.normal(0, 1, (V, d)).astype(np.float32)
    dOut = rng.normal(0, 1, (V, d)).astype(np.float32)
    w = {"W_forward": rng.normal(0, 0.3, (R, B, s, s)).astype(np.float32),
         "W_backward": rng.normal(0, 0.3, (R, B, s, s)).astype(np.float32),
         "W_self": rng.normal(0, 0.05, (d, d)).astype(np.float32)}
    for k in ("W_forward", "W_backward"):
        w[k][unused] = 0
    cu = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    poisoned = {k: v.copy() for k, v in w.items()}
    for k in ("W_forward", "W_backward"):
        poisoned[k][unused] = np.nan

    def fn():
        Ht = cu(H).requires_grad_(True)
        Wf, Wb, Ws = (cu(poisoned[k]).requires_grad_(True) for k in ("W_forward", "W_backward", "W_self"))
        out = ops.block_layer(Ht, Wf, Wb, Ws, g, B, None, 1.0, False)
        out.backward(cu(dOut))
        return out.detach(), {"H": Ht.grad, "W_forward": Wf.grad, "W_backward": Wb.grad, "W_self": Ws.grad}

    (out, grads), names = traced_kernels(fn)
    r_out, r_g = oracle.layer_fwd_bwd("block", H, tr, w, nf, nb, dOut, None, 1.0, False, torch.float64)
    a_out, a_g = oracle.layer_fwd_bwd("block", np.abs(H), tr, {k: np.abs(v) for k, v in w.items()}, nf, nb,
                                      np.abs(dOut), None, 1.0, False, torch.float64)
    check(case, "out", out, r_out, a_out)
    for k in grads:
        check(case, "d" + k, grads[k], r_g[k], a_g[k])
    for k in ("W_forward", "W_backward"):
        assert (grads[k][unused] == 0).all(), "d%s of the unused relation" % k
    return names


def run_basis(case, item_max):
    rng = np.random.RandomState(zlib.crc32(case.name.encode()))
    d, B = case.d, case.B
    V, R, unused = 3 * ST - 40, 6, 4
    tr, nf, nb, g = layer_graph(rng, V, R, unused, item_max)
    H = rng.normal(0, 1, (V, d)).astype(np.float32)
    dOut = rng.normal(0, 1, (V, d)).astype(np.float32)
    sd = 1.0 / np.sqrt(d)
    w = {"W_forward": rng.normal(0, sd, (d, B, d)).astype(np.float32),
         "W_backward": rng.normal(0, sd, (d, B, d)).astype(np.float32),
         "C_forward": rng.normal(0, 1, (R, B)).astype(np.float32),
         "C_backward": rng.normal(0, 1, (R, B)).astype(np.float32),
         "W_self": rng.normal(0, sd, (d, d)).astype(np.float32)}
    for k in ("C_forward", "C_backward"):
        w[k][unused] = 0
    poisoned = {k: v.copy() for k, v in w.items()}
    for k in ("C_forward", "C_backward"):
        poisoned[k][unused] = np.nan
    cu = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    names_ = ("W_forward", "W_backward", "C_forward", "C_backward", "W_self")

    def fn():
        Ht = cu(H).requires_grad_(True)
        ts = [cu(poisoned[k]).requires_grad_(True) for k in names_]
        out = ops.basis_layer(Ht, *ts, g, None, 1.0, False)
        out.backward(cu(dOut))
        grads = {"H": Ht.grad}
        grads.update({k: t.grad for k, t in zip(names_, ts)})
        return out.detach(), grads

    (out, grads), names = traced_kernels(fn)
    r_out, r_g = oracle.layer_fwd_bwd("basis", H, tr, w, nf, nb, dOut, None, 1.0, False, torch.float64)
    a_out, a_g = oracle.layer_fwd_bwd("basis", np.abs(H), tr, {k: np.abs(v) for k, v in w.items()}, nf, nb,
                                      np.abs(dOut), None, 1.0, False, torch.float64)
    check(case, "out", out, r_out, a_out)
    for k in grads:
        check(case, "d" + k, grads[k], r_g[k], a_g[k])
    for k in ("C_forward", "C_backward"):
        assert (grads[k][unused] == 0).all(), "d%s of the unused relation" % k
    return names


def run_gemm(case, item_max):
    g = torch.Generator(device=DEV).manual_seed(3)
    M, N, K = 300, 132, 100
    A = torch.randn(M, K, device=DEV, generator=g)
    Bm = torch.randn(K, N, device=DEV, generator=g)
    if case.entry == "gemm":
        C, names = traced_kernels(lambda: ops.gemm_tf32x3(A, Bm))
        ref, absref = A.double().cpu() @ Bm.double().cpu(), A.double().abs().cpu() @ Bm.double().abs().cpu()
    else:
        At = torch.randn(K, M - 44, device=DEV, generator=g)
        C, names = traced_kernels(lambda: ops.gemm_tn_tf32x3(At, Bm))
        ref, absref = At.double().cpu().T @ Bm.double().cpu(), At.double().abs().cpu().T @ Bm.double().abs().cpu()
    check(case, "C", C, ref, absref)
    return names


def run_rank(case, item_max):
    """Integer codes: every energy is exact, so the ranks must equal the numpy count exactly."""
    rng = np.random.RandomState(4)
    V, d, n = 1000, 64, 200
    codes = (rng.randint(-1, 2, (V, d)) * (rng.uniform(size=(V, d)) < 0.1)).astype(np.float32)
    relt = rng.randint(-1, 2, (V, d)).astype(np.float32)
    X = np.stack([rng.randint(0, V, n), rng.randint(0, V, n), rng.randint(0, V, n)], 1).astype(np.int32)
    ranker = ops.DistMultRanker(torch.as_tensor(codes, device=DEV), torch.as_tensor(relt, device=DEV))
    (raw, _), names = traced_kernels(lambda: ranker.rank(torch.as_tensor(X, device=DEV), 1, None))
    e = (codes[X[:, 0]].astype(np.float64) * relt[X[:, 1]]) @ codes.T.astype(np.float64)
    ref = (e >= e[np.arange(n), X[:, 2]][:, None]).sum(1)
    np.testing.assert_array_equal(raw.cpu().numpy(), ref)
    return names


RUNNERS = {"agg": run_agg, "layer": run_layer, "basis": run_basis, "gemm": run_gemm, "tn": run_gemm,
           "rank": run_rank}


@pytest.fixture(autouse=True)
def restore_block_algo():
    yield
    _lib.set_option("block_algo", -1)


def test_profiler_sees_library_kernels():
    """Canary: the library links its own CUDA runtime; its kernels must still show up in a torch.profiler trace,
    or no expectation below could be checked."""
    A = torch.randn(256, 64, device=DEV)
    Bm = torch.randn(64, 128, device=DEV)
    _, names = traced_kernels(lambda: ops.gemm_tf32x3(A, Bm))
    assert {"k_split_b", "k_gemm_tf32x3<0>"} <= names, sorted(names)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_kernel_instantiation_vs_float64(case, monkeypatch):
    monkeypatch.setenv("RGCN_SUPERTILE_ROWS", str(ST))
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    item_max = int(case.env.get("RGCN_ITEM_MAX", ITEM_MAX))
    _lib.set_option("block_algo", case.algo)
    names = RUNNERS[case.entry](case, item_max)
    missing = [k for k in case.expect if k not in names]
    assert not missing, "%s: expected kernels not in the trace: %s; traced: %s" % (
        case.name, missing, sorted(n for n in names if n.split("<")[0] in {e.split("<")[0] for e in case.expect}))
    worst = max((v for (c, _), v in WORST.items() if c == case.name), default=0.0)
    print("%s: worst elementwise |err|/absref %.3e" % (case.name, worst))
