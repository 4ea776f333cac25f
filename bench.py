#!/usr/bin/env python
"""bench.py -- R-GCN layer fwd+bwd throughput (M-edges/s) on B200, one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--scale S] [--impl ours|reference]
                  [--dump-outputs DIR]

A "step" is ONE pass of the hot path over one graph: one block-diagonal R-GCN layer forward + backward
(dH, dW_forward, dW_backward, dW_self) on synthetic data of the named shape.  K timed steps follow W warm-up steps.
--dump-outputs DIR writes what the last timed step returned (out, dH, dW_forward, dW_backward, dW_self) as
DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs (see dump_outputs).
Metric (BASELINE.json): M-edges/s = triples E / (t_fwd + t_bwd) / 1e6, graph prep excluded from `value`
(device-resident inputs) and INCLUDED in `e2e` (host buffers in, host buffers out).

Workloads
  synthetic  (DEFAULT; BASELINE configs[4], the configuration north_star's targets are quoted on) V = 10 M x scale,
             R = 1000, E = 100 M x scale, d = 512, B = 64 (s = 8), uniform endpoints: the HBM-bound regime.
             --scale defaults to the largest of {1, 0.5, 0.25, 0.1, 0.05, 0.02} whose working set fits the GPU
             (1.0 = the full 10 M-node / 100 M-edge graph needs ~135 GB of the B200's 180 GB) and is named in
             config.workload.  --gpus N shards THE SAME graph over N GPUs: strong scaling.
  fb15k237   (secondary, BASELINE configs[1]) V=14541 R=237 E=272115, d=500, B=100 (s=5): the FB15k-237
             evaluation graph shape of settings/gcn_block.exp, synthetic skewed KG; cache-resident (H = 29 MB).
             --gpus N grows the graph with N (weak scaling of a toy-sized shard), kept for continuity with round 1.
  fb15k237-train  the E = 15000 train-step graph of the same configuration.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCALES = (1.0, 0.5, 0.25, 0.1, 0.05, 0.02)


def synthetic_kg(V, R, E, seed=1234, skewed=False):
    """SURVEY.md 8(d) generator (PCG64(seed)): uniform, or skewed s,o = floor(V*u^3) under a fixed
    random relabelling and r = floor(R*u^2)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if not skewed:
        s = rng.integers(0, V, E, dtype=np.int32)
        o = rng.integers(0, V, E, dtype=np.int32)
        r = rng.integers(0, R, E, dtype=np.int32)
    else:
        perm = rng.permutation(V)
        s = perm[np.minimum((V * rng.random(E) ** 3).astype(np.int64), V - 1)]
        o = perm[np.minimum((V * rng.random(E) ** 3).astype(np.int64), V - 1)]
        r = np.minimum((R * rng.random(E) ** 2).astype(np.int64), R - 1)
    out = np.empty((E, 3), np.int32)
    out[:, 0], out[:, 1], out[:, 2] = s, r, o
    return out


def working_set_bytes(V, E, d, R, s, world=1):
    """Peak device bytes of one rank of the timed step (features, gradients, workspace, graph views, prep scratch)."""
    Vl, Ml = V // world, 2 * E // world
    halo = 0 if world == 1 else min(V - Vl, Ml)          # unique remote sources (uniform graph: nearly all of them)
    feat = (4 * Vl + 2 * Vl + 4 * halo) * d * 4           # H, dOut, out, dH | G, dS | halo rows in/out + send/back
    graph = Ml * (2 * 12 + 28) + (3 * 2 * E * 4 if world > 1 else 0)
    return feat + graph + 3 * 2 * R * s * d * 4 + (1 << 30)


def pick_scale(args, total_mem, world):
    if args.scale is not None:
        return args.scale
    for sc in SCALES:
        if working_set_bytes(int(10_000_000 * sc), int(100_000_000 * sc), 512, 1000, 8, world) <= 0.88 * total_mem:
            return sc
    return SCALES[-1]


def workload_spec(args, world, scale=None):
    if args.workload == "fb15k237":
        return dict(name="fb15k237-evalgraph gcn_block d=500 B=100 (BASELINE configs[1])", V=14541 * world, R=237,
                    E=272115 * world, d=500, B=100, skewed=True, scaling="weak")
    if args.workload == "fb15k237-train":
        return dict(name="fb15k237 train-step graph E=15000 gcn_block d=500 B=100", V=14541 * world, R=237,
                    E=15000 * world, d=500, B=100, skewed=True, scaling="weak")
    if args.workload == "synthetic":
        sc = scale if scale is not None else (args.scale if args.scale is not None else 1.0)
        V, E = int(10_000_000 * sc), int(100_000_000 * sc)
        full = "the full graph" if sc == 1.0 else "x%.3g of it (largest scale whose working set fits)" % sc
        return dict(name="synthetic KG 10M nodes / 1k relations / 100M edges d=512 B=64 (BASELINE configs[4]): %s, "
                         "V=%d E=%d" % (full, V, E), V=V, R=1000, E=E, d=512, B=64, skewed=args.skewed,
                    scaling="strong", scale=sc)
    raise SystemExit("unknown workload " + args.workload)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            j = json.load(fh)
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                               f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:  # region shorter than one sample: take whatever was seen
            for ts, line in self.rows[-3:]:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0]))
                    mx.append(float(f[1]))
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_sample_spec(spec, sample_E):
    """The CPU arms run a BOUNDED sample of the workload: `sample_E` triples of the same generator with the same R,
    d, B.  For the synthetic workload the node set shrinks with the edges (same 10 edges per node), because the
    restated reference materialises [V, d] feature matrices (20 GB at V = 10 M); the FB shapes keep their V."""
    V = spec["V"]
    if spec.get("scaling") == "strong":
        V = max(1000, sample_E // 10)
    return dict(spec, V=V, E=sample_E)


def oracle_step_factory(spec, sample_E, seed=0, return_inputs=False):
    """The reference's CPU path restated (oracle/rgcn_oracle.py), on a bounded sample of the workload."""
    import torch

    from oracle import rgcn_oracle as oracle
    torch.set_num_threads(os.cpu_count() or 1)
    sp = cpu_sample_spec(spec, sample_E)
    V, R, d, B = sp["V"], sp["R"], sp["d"], sp["B"]
    tr = synthetic_kg(V, R, sample_E, seed=1234, skewed=sp["skewed"])
    rng = np.random.RandomState(seed)
    H = rng.normal(0, 1, (V, d)).astype(np.float32)
    dOut = rng.normal(0, 1, (V, d)).astype(np.float32)
    w = oracle.init_block_layer(rng, R, d, B)
    nf, nb = oracle.graph_norms(tr, V)

    def step(dtype=torch.float32):
        return oracle.layer_fwd_bwd("block", H, tr, w, nf, nb, dOut, None, 1.0, True, dtype)
    if return_inputs:
        return step, dict(V=V, R=R, d=d, B=B, triples=tr, H=H, dOut=dOut, w=w)
    return step


def time_cpu(step, steps, warmup):
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps


def best_cpu_threads(step):
    """The restated reference is memory/launch bound: more torch threads than ~16-32 SLOW it down on
    a many-core host.  Give the baseline its best configuration: try a few counts, keep the fastest."""
    import torch
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    step()  # warm-up (allocator, thread pool)
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        step()
        t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  TensorFlow 1.4 cannot be
    installed here (no wheel for py3.12, no network), so this times the oracle port (the one other
    place bench.py may execute oracle/), all host threads, on a bounded sample of our arm's config."""
    if rank != 0:
        return
    spec = workload_spec(args, 1)
    sample_E = min(spec["E"], args.cpu_sample_edges)
    step = oracle_step_factory(spec, sample_E)
    cores = best_cpu_threads(step)
    # keep the whole --steps K run within a few minutes: shrink the per-step sample if K steps of it would not
    est = time_cpu(step, 1, 1)
    budget_s = 150.0
    if est * args.steps > budget_s and sample_E > 2000:
        sample_E = max(2000, int(sample_E * budget_s / (est * args.steps)))
        step = oracle_step_factory(spec, sample_E)
    sec = time_cpu(step, args.steps, max(1, min(args.warmup, 1)))
    val = sample_E / sec / 1e6
    sp = cpu_sample_spec(spec, sample_E)
    sample = "%d triples over %d nodes of the same generator (same R, d, B; ours runs E=%d, V=%d), fp32, best of {8,16,32,64,all} torch threads = %d of %d host cores" % (
        sample_E, sp["V"], spec["E"], spec["V"], cores, os.cpu_count() or 1)
    line = {"impl": "reference", "metric": "R-GCN layer fwd+bwd M-edges/sec", "value": val,
            "unit": "M-edges/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": spec["name"], "V": sp["V"], "R": spec["R"], "E": sample_E,
                       "d": spec["d"], "B": spec["B"],
                       "note": "reference TF1 CPU path restated op-for-op in torch-CPU (TensorFlow 1.4 not installable); "
                               "bounded sample, per-edge normalised"},
            "cpu_baseline": {"value": val, "unit": "M-edges/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "M-edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def lib_stamp():
    p = os.path.join(ROOT, "relationprediction_b200", "lib", "librgcn_b200.stamp")
    try:
        with open(p) as fh:
            return fh.read().strip()[:16]
    except OSError:
        return None


def kernel_source_stamp():
    """Fingerprint of the sources of the aggregation kernels whose DRAM traffic profiles/r2_traffic.json records
    (csrc/block_staged.cu + csrc/kernels.cuh): the traffic entry is stale when THESE change, not when any other part
    of the library does."""
    import hashlib
    h = hashlib.sha256()
    for name in ("block_staged.cu", "kernels.cuh"):
        try:
            with open(os.path.join(ROOT, "relationprediction_b200", "csrc", name), "rb") as fh:
                h.update(fh.read())
        except OSError:
            return None
    return h.hexdigest()[:16]


def relerr(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


DUMP_BYTES_PER_ARRAY = 12 << 20   # five arrays: at most 60 MiB per dump


def dump_outputs(outdir, arrays):
    """Writes each tensor as float32 <outdir>/<name>.npy.  A tensor larger than DUMP_BYTES_PER_ARRAY is replaced by a
    fixed sample of its rows (first dimension): the sorted indices np.random.default_rng(0).choice(rows, k,
    replace=False) with k = DUMP_BYTES_PER_ARRAY // row bytes, the same rows in every run of the same shape."""
    import torch
    os.makedirs(outdir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        rows = t.shape[0]
        k = max(1, DUMP_BYTES_PER_ARRAY // (t[0].numel() * 4))
        if k < rows:
            idx = np.sort(np.random.default_rng(0).choice(rows, k, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(outdir, name + ".npy"), t.cpu().numpy())


def parity_check_sharded(rank, world, dev, B, d, R, transport=None):
    """N > 1: a small graph through the SAME sharded code path (device plan, overlapped halo exchange, gradient
    all-reduce) against the single-GPU layer computed on rank 0.  The driver's GPU test box has one GPU, so this is
    where the 4- and 8-rank equivalence is verified every time the scaling bench runs."""
    import torch
    import torch.distributed as dist

    from relationprediction_b200 import ops, parallel
    V, E = 8 * 1500, 120000
    tr = synthetic_kg(V, R, E, seed=77, skewed=True)
    tri = torch.from_numpy(tr).to(dev)
    s = d // B
    gen = torch.Generator(device=dev).manual_seed(5)   # same seed on every rank: replicated inputs
    H = torch.randn(V, d, device=dev, generator=gen)
    dOut = torch.randn(V, d, device=dev, generator=gen)
    ws = [torch.randn(R, B, s, s, device=dev, generator=gen) * 0.2, torch.randn(R, B, s, s, device=dev, generator=gen) * 0.2,
          torch.randn(d, d, device=dev, generator=gen) * 0.05]
    sg = parallel.ShardedGraph(tri, V, R, rank, world, dev, transport=transport)
    p = sg.plan
    Hl = H[p.lo:p.hi].clone().requires_grad_(True)
    wl = [w.clone().requires_grad_(True) for w in ws]
    out = sg.block_layer(Hl, wl[0], wl[1], wl[2], B, None, 1.0, True)
    out.backward(dOut[p.lo:p.hi].contiguous())
    sg.allreduce_weight_grads(wl)
    n_max = max(parallel.node_bounds(V, world)[i + 1] - parallel.node_bounds(V, world)[i] for i in range(world))
    pad = lambda t: torch.cat([t, t.new_zeros(n_max - t.shape[0], t.shape[1])]) if t.shape[0] < n_max else t
    outs = [torch.empty(n_max, d, device=dev) for _ in range(world)]
    dhs = [torch.empty(n_max, d, device=dev) for _ in range(world)]
    dist.all_gather(outs, pad(out.detach()))
    dist.all_gather(dhs, pad(Hl.grad))
    res = None
    if rank == 0:
        b = parallel.node_bounds(V, world)
        out_all = torch.cat([outs[i][:b[i + 1] - b[i]] for i in range(world)])
        dh_all = torch.cat([dhs[i][:b[i + 1] - b[i]] for i in range(world)])
        g1 = ops.Graph.from_device_triples(tri, V, R)
        H1 = H.clone().requires_grad_(True)
        w1 = [w.clone().requires_grad_(True) for w in ws]
        o1 = ops.block_layer(H1, w1[0], w1[1], w1[2], g1, B, None, 1.0, True)
        o1.backward(dOut)
        errs = {"out": relerr(out_all, o1.detach()), "dH": relerr(dh_all, H1.grad),
                "dW_forward": relerr(wl[0].grad, w1[0].grad), "dW_backward": relerr(wl[1].grad, w1[1].grad),
                "dW_self": relerr(wl[2].grad, w1[2].grad)}
        res = {"what": "sharded (this N, %s transport) vs single-GPU layer on rank 0, skewed KG V=%d E=%d d=%d B=%d"
                       % (sg.halo_transport() or "nccl", V, E, d, B),
               "max_rel_err": max(errs.values()), "rel_err": errs, "tolerance": 1e-5,
               "ok": bool(max(errs.values()) <= 1e-5)}
    dist.barrier()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="synthetic", choices=["synthetic", "fb15k237", "fb15k237-train"])
    ap.add_argument("--scale", type=float, default=None,
                    help="synthetic workload: fraction of 10M nodes / 100M edges (default: the largest that fits)")
    ap.add_argument("--skewed", action="store_true", help="synthetic workload: skewed endpoints")
    ap.add_argument("--cpu-sample-edges", type=int, default=20000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (needs 4 pinned V*d buffers)")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--shard", choices=["node", "feature"], default="node",
                    help="N > 1: 1-D node shard with halo all-to-all (default, north_star) or the experimental "
                         "feature-sharded message passing (replicated graph, two transposes per layer)")
    ap.add_argument("--halo", choices=["overlapped", "pipelined"], default="overlapped",
                    help="N > 1, node shard: one all-to-all per layer direction overlapped with the local-source work "
                         "(default) or the per-peer ring that aggregates peer k's rows while peer k+1's are in flight")
    ap.add_argument("--transport", choices=["auto", "peer", "nccl"], default="auto",
                    help="N > 1, overlapped halo exchange: 'peer' = rows pushed into peer-mapped halo buffers by "
                         "rgcn_rows_gather over NVLink, 'nccl' = packed rows + all-to-all; auto = peer, NCCL when "
                         "symmetric memory cannot be set up")
    ap.add_argument("--triples-npz", default=None,
                    help="use the triples of this .npz (arrays: triples [E,3], V, R) instead of the synthetic generator; "
                         "diagnostic only (e.g. the real FB15k-237 graph), the default bench stays synthetic")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's out, dH and weight gradients to "
                         "DIR/<name>.npy (float32; a fixed row sample of any array over 12 MiB); with N > 1 each rank "
                         "writes its own under DIR/rank<r>/")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))

    import torch
    import torch.distributed as dist

    from relationprediction_b200 import _lib, ops
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    total_mem = torch.cuda.get_device_properties(dev).total_memory

    scale = pick_scale(args, total_mem, world) if args.workload == "synthetic" else None
    spec = workload_spec(args, world, scale)
    V, R, E, d, B = spec["V"], spec["R"], spec["E"], spec["d"], spec["B"]
    s = d // B
    strong = spec["scaling"] == "strong"
    if args.triples_npz:
        z = np.load(args.triples_npz)
        triples = np.ascontiguousarray(z["triples"], dtype=np.int32)
        V, R, E = int(z["V"]), int(z["R"]), int(triples.shape[0])
        spec = dict(spec, name="triples from " + os.path.basename(args.triples_npz), V=V, R=R, E=E)
    else:
        triples = synthetic_kg(V, R, E, seed=1234, skewed=spec["skewed"])
    tri_dev = torch.from_numpy(triples).to(dev)
    if E > 20_000_000:
        triples = None   # the host copy is only kept for the e2e leg of small workloads

    # the block-diagonal benchmark walks the weight-id-major views only (deterministic mode needs the CSR views too)
    if os.environ.get("RGCN_BLOCK_ALGO") != "0":
        _lib.set_option("graph_views", 2)

    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if world == 1:
        graph = ops.Graph.from_device_triples(tri_dev, V, R)
        layer = None
        V_loc = V
    else:
        from relationprediction_b200 import parallel
        if args.shard == "feature":   # experimental: replicated graph, messages feature-parallel (parallel.py)
            layer = parallel.FeatureShardedGraph(tri_dev.cpu().numpy(), V, R, rank, world, dev, B, s)
            graph = layer.graph
        else:
            layer = parallel.ShardedGraph(tri_dev, V, R, rank, world, dev, pipelined=(args.halo == "pipelined"),
                                          transport=None if args.transport == "auto" else args.transport)
            graph = layer.graph_local
        V_loc = layer.n_local
    torch.cuda.synchronize()
    prep_ms = (time.perf_counter() - t0) * 1e3
    info = graph.info()
    if E > 20_000_000:
        del tri_dev
        tri_dev = None

    H = torch.randn(V_loc, d, device=dev, generator=gen).requires_grad_(True)
    dOut = torch.randn(V_loc, d, device=dev, generator=gen)
    std = 3.0 / np.sqrt(R + s)  # glorot_variance([R, s]) used as std (gcn_basis_concat.py:22)
    wgen = torch.Generator(device=dev).manual_seed(2)  # replicated weights: same seed on every rank
    Wf = (torch.randn(R, B, s, s, device=dev, generator=wgen) * std).requires_grad_(True)
    Wb = (torch.randn(R, B, s, s, device=dev, generator=wgen) * std).requires_grad_(True)
    Ws = (torch.randn(d, d, device=dev, generator=wgen) * std).requires_grad_(True)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step(h=None, do=None):
        h = H if h is None else h
        for t in (h, Wf, Wb, Ws):
            t.grad = None
        if world == 1:
            out = ops.block_layer(h, Wf, Wb, Ws, graph, B, None, 1.0, True)
            out.backward(dOut if do is None else do)
        else:
            out = layer.block_layer(h, Wf, Wb, Ws, B, None, 1.0, True)
            out.backward(dOut if do is None else do)
            layer.allreduce_weight_grads([Wf, Wb, Ws])
        return out

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None  # started early: nvidia-smi needs ~0.3 s to emit
    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()

    def timed_region():
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        l0 = _lib.launch_count()
        sync_all()
        w0 = time.time()
        last_out = None
        for i in range(args.steps):
            flush_buf.zero_()  # L2 flush between timed iterations (outside the event pair)
            ev0[i].record()
            if i + 1 < args.steps:
                step()
            else:
                last_out = step()   # kept for --dump-outputs; earlier outputs are freed as they come
            ev1[i].record()
        sync_all()
        w1 = time.time()
        ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, w0, w1, _lib.launch_count() - l0, last_out

    total_ms, wall0, wall1, launches, last_out = timed_region()
    clocks = sampler.stop(wall0, wall1) if sampler else None
    remeasured = False
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    flag = torch.tensor([1 if (clocks and bad & set(clocks.get("reasons", []))) else 0], device=dev)
    if world > 1:
        dist.broadcast(flag, src=0)
    if int(flag.item()):  # a throttled run is rejected and re-measured once (B200_PROFILING.md)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        time.sleep(0.5)
        last_out = None
        total_ms, wall0, wall1, launches, last_out = timed_region()
        clocks = sampler.stop(wall0, wall1) if sampler else None
        remeasured = True
    if clocks is not None:
        clocks["remeasured_after_throttle"] = remeasured
    ms_per_step = total_ms / args.steps
    value = E / (ms_per_step * 1e-3) / 1e6
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, "rank%d" % rank),
                     {"out": last_out, "dH": H.grad, "dW_forward": Wf.grad, "dW_backward": Wb.grad,
                      "dW_self": Ws.grad})
    last_out = None   # at full scale the output is 20 GB: released before the profiling and e2e legs

    # ---- per-stage timing (separate pass, events inside the library): roofline of the dominant kernel and of the layer
    peak, peak_src = peaks()
    wt_bytes = 2 * R * s * d * 4 + 4 * d * d            # SURVEY 8(d) Wbytes: both block tables + W_self
    roofline, roofline_layer, stages = None, None, None
    n_prof = 3 if E > 20_000_000 else 5
    prof_ok = False
    if rank == 0:
        try:
            _lib.profile_enable(True)
            prof_ok = True
        except Exception as exc:  # noqa: BLE001
            stages = {"error": repr(exc)}
    for _ in range(n_prof):          # identical and unguarded on every rank (the steps contain collectives)
        flush_buf.zero_()
        step()
        torch.cuda.synchronize()
    if rank == 0 and prof_ok:
        try:
            acc = {}
            for name, ms in _lib.profile_read():
                acc[name] = acc.get(name, 0.0) + ms / n_prof
            _lib.profile_enable(False)
            stages = {k: round(v, 5) for k, v in acc.items()}
            if world == 1:
                M = 2 * E
                alg = {"block_agg_fwd": M * (4 * d + 12) + 8 * V * d + 2 * R * s * d * 4,
                       "block_agg_dH": M * (8 * d + 12) + 8 * V * d + 4 * R * s * d * 4,
                       "block_dW": M * (8 * d + 12) + 4 * R * s * d * 4}
                if acc.get("block_dW", 1.0) < 0.02:   # dW was produced inside the dH walk (fused kernel)
                    alg.pop("block_dW")
                else:
                    alg["block_agg_dH"] = M * (4 * d + 12) + 8 * V * d + 2 * R * s * d * 4
            elif args.shard == "feature":   # every rank walks ALL messages on d_local-wide rows
                M_all, dl, Vn = layer.graph.M, layer.d_local, layer.n_nodes
                wq = 2 * R * s * dl * 4
                alg = {"block_aggregate": M_all * (4 * dl + 12) + 4 * Vn * dl + wq,
                       "block_aggregate_bwd": M_all * (8 * dl + 12) + 4 * Vn * dl + 2 * wq}
            else:
                M_loc, M_halo = layer.graph_local.M, layer.graph_halo.M
                wq = 2 * R * s * d * 4
                alg = {"block_agg_fwd": M_loc * (4 * d + 12) + 8 * V_loc * d + wq,
                       "block_aggregate": M_halo * (4 * d + 12) + 4 * V_loc * d + wq,
                       "block_agg_dH": M_loc * (8 * d + 12) + 8 * V_loc * d + 2 * wq,
                       "block_aggregate_bwd": M_halo * (8 * d + 12) + 4 * layer.n_halo * d + 2 * wq}
            mine = {k: v for k, v in acc.items() if k in alg and v > 0}
            if mine:
                top = max(mine, key=mine.get)
                achieved = alg[top] / (mine[top] * 1e-3) / 1e9
                traffic, stale = None, None
                tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
                if os.path.exists(tp) and world == 1:
                    with open(tp) as fh:
                        tj = json.load(fh)
                    ent = tj.get("%s|%s" % (args.workload, spec.get("scale", "")), {})
                    traffic = ent.get(top)
                    stale = bool(ent.get("kernel_source_stamp") != kernel_source_stamp()) if traffic is not None else None
                roofline = {"kernel": top + (" (rank 0 shard)" if world > 1 else ""), "bound": "hbm", "achieved": achieved,
                            "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                            "traffic_stale": stale,
                            "traffic_source": "profiles/r2_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one "
                                              "ncu --set full launch of this kernel on this workload" if traffic else None,
                            "algorithmic_bytes": int(alg[top]), "kernel_ms": mine[top], "peak_source": peak_src,
                            "all": {k: {"ms": mine[k], "GB/s": alg[k] / (mine[k] * 1e-3) / 1e9,
                                        "frac": alg[k] / (mine[k] * 1e-3) / 1e9 / peak} for k in mine}}
        except Exception as exc:  # noqa: BLE001
            roofline, stages = None, {"error": repr(exc)}
    # layer level (what north_star's ">= 60 % on the fused layer" asks): SURVEY 8(d) fwd+bwd = 2E(12d+24) + 24Vd + 3 Wbytes,
    # whole job, against N x the measured per-GPU peak
    layer_bytes = 2 * E * (12 * d + 24) + 24 * V * d + 3 * wt_bytes
    layer_ach = layer_bytes / (ms_per_step * 1e-3) / 1e9
    roofline_layer = {"bound": "hbm", "algorithmic_bytes": int(layer_bytes), "achieved": layer_ach, "unit": "GB/s",
                      "peak": peak * world, "frac": layer_ach / (peak * world), "peak_source": peak_src,
                      "formula": "2E(12d+24) + 24Vd + 3(8Rds + 4d^2) bytes / ms_per_step (SURVEY.md 8d), whole job over N GPUs"}
    sync_all()

    # ---- N > 1: equivalence sharded == single GPU on a small graph, every run ----
    parity = None
    if world > 1 and args.shard == "node" and not args.no_parity_check:
        try:
            parity = parity_check_sharded(rank, world, dev, B, d, R,
                                          transport=None if args.transport == "auto" else args.transport)
        except Exception as exc:  # noqa: BLE001  (every rank takes the same path: the check has no data-dependent branch)
            parity = {"error": repr(exc)}
        sync_all()

    # ---- e2e: same layer fwd+bwd through the public API with HOST buffers ----
    # Every step: pinned host buffers -> H2D -> (N = 1: GPU graph prep from the host edge list) -> fwd -> bwd ->
    # D2H of out, dH and the weight gradients.  The resident benchmark tensors are released first: at full size
    # the e2e leg needs the memory for its own device copies.
    e2e = None
    if not args.no_e2e:
        H_pin = H.detach().cpu().pin_memory()
        dOut_pin = dOut.cpu().pin_memory()
        out_host = torch.empty(V_loc, d).pin_memory()
        dH_host = torch.empty(V_loc, d).pin_memory()
        dW_host = [torch.empty_like(t, device="cpu").pin_memory() for t in (Wf, Wb, Ws)]
        tri_pin = None
        if world == 1:
            tri_pin = (torch.from_numpy(triples) if triples is not None else
                       torch.from_numpy(synthetic_kg(V, R, E, seed=1234, skewed=spec["skewed"]))).pin_memory()
            del graph
            graph = None
        del H, dOut
        H = dOut = None
        torch.cuda.empty_cache()
        h2d = (H_pin.numel() + dOut_pin.numel()) * 4 + (tri_pin.numel() * 4 if tri_pin is not None else 0)
        d2h = (out_host.numel() + dH_host.numel() + sum(t.numel() for t in dW_host)) * 4
        prep_times = []
        copy_stream = torch.cuda.Stream(device=dev)

        def e2e_step():
            with torch.cuda.stream(copy_stream):  # feature / gradient inputs on a side stream, concurrently with graph prep
                h = H_pin.to(dev, non_blocking=True)
                do = dOut_pin.to(dev, non_blocking=True)
            in_ready = copy_stream.record_event()
            if world == 1:
                tp = time.perf_counter()
                g2 = ops.Graph.from_device_triples(tri_pin.to(dev, non_blocking=True), V, R)  # H2D + GPU graph prep
                prep_times.append(time.perf_counter() - tp)
            torch.cuda.current_stream().wait_event(in_ready)
            h.requires_grad_(True)
            for t in (Wf, Wb, Ws):
                t.grad = None
            if world == 1:
                o = ops.block_layer(h, Wf, Wb, Ws, g2, B, None, 1.0, True)
            else:
                o = layer.block_layer(h, Wf, Wb, Ws, B, None, 1.0, True)
            fwd_done = torch.cuda.current_stream().record_event()
            with torch.cuda.stream(copy_stream):  # D2H of the forward result overlaps the backward pass
                copy_stream.wait_event(fwd_done)
                out_host.copy_(o.detach(), non_blocking=True)
            o.backward(do)
            if world > 1:
                layer.allreduce_weight_grads([Wf, Wb, Ws])
            dH_host.copy_(h.grad, non_blocking=True)
            for hh, t in zip(dW_host, (Wf, Wb, Ws)):
                hh.copy_(t.grad, non_blocking=True)
            torch.cuda.synchronize()

        n_e2e = 3 if E > 20_000_000 else max(3, min(args.steps, 10))
        e2e_step()
        prep_times.clear()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        sync_all()
        e2e_ms = (time.perf_counter() - t0) / n_e2e * 1e3
        if world > 1:
            tt = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_ms = float(tt.item())
        e2e = {"value": E / (e2e_ms * 1e-3) / 1e6, "unit": "M-edges/s", "h2d_bytes_per_step": int(h2d) * world,
               "d2h_bytes_per_step": int(d2h) * world, "ms_per_step": e2e_ms, "steps": n_e2e,
               "what": ("pinned host buffers every step: triples -> GPU graph prep || H2D(H, dOut) -> fwd -> bwd || "
                        "D2H(out) -> D2H(dH, dW*); one device sync at the end") if world == 1 else
                       ("per rank: pinned host H/dOut shard -> H2D -> sharded fwd+bwd (halo exchange, grad all-reduce) "
                        "-> D2H(out, dH shard, dW*); the shard plan + graph handles are built once (graph prep per step is "
                        "measured in the single-GPU e2e)")}
        if prep_times:
            e2e["host_graph_prep_ms"] = float(np.mean(prep_times) * 1e3)

    # ---- CPU baseline (rank 0): the restated reference on a bounded sample; the same sample through the GPU path
    #      is compared with the oracle's float64 result (the oracle as the checker)
    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        spec1 = workload_spec(args, 1, scale)
        sample_E = min(spec1["E"], args.cpu_sample_edges)
        cstep, inp = oracle_step_factory(spec1, sample_E, return_inputs=True)
        used = best_cpu_threads(cstep)
        sec = time_cpu(cstep, 3, 0)
        cpu_baseline = {"value": sample_E / sec / 1e6, "unit": "M-edges/s", "cores": used,
                        "host_cores": os.cpu_count() or 1, "kind": "port",
                        "sample": "%d triples over %d nodes of the same generator (same R, d, B), 3 timed fwd+bwd passes of "
                                  "the torch-CPU restatement (TensorFlow 1.4 not installable)" % (sample_E, inp["V"])}
        if not args.no_parity_check:
            try:
                ref_out, ref_g = cstep(torch.float64)
                _lib.set_option("graph_views", 3)
                g3 = ops.Graph(inp["triples"], inp["V"], inp["R"], device=local_rank)
                ht = torch.from_numpy(inp["H"]).to(dev).requires_grad_(True)
                wt3 = [torch.from_numpy(inp["w"][k]).to(dev).requires_grad_(True) for k in ("W_forward", "W_backward", "W_self")]
                o3 = ops.block_layer(ht, wt3[0], wt3[1], wt3[2], g3, inp["B"], None, 1.0, True)
                o3.backward(torch.from_numpy(inp["dOut"]).to(dev))
                errs = {"out": relerr(o3.detach().cpu().double(), ref_out), "dH": relerr(ht.grad.cpu().double(), ref_g["H"])}
                for t, k in zip(wt3, ("W_forward", "W_backward", "W_self")):
                    errs["d" + k] = relerr(t.grad.cpu().double(), ref_g[k])
                cpu_baseline["parity_vs_oracle_f64"] = {"max_rel_err": max(errs.values()), "rel_err": errs,
                                                        "tolerance": 1e-4, "ok": bool(max(errs.values()) <= 1e-4)}
            except Exception as exc:  # noqa: BLE001
                cpu_baseline["parity_vs_oracle_f64"] = {"error": repr(exc)}

    if rank == 0:
        line = {"metric": "R-GCN layer fwd+bwd M-edges/sec", "value": value, "unit": "M-edges/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
                "dtype": "f32", "data": "synthetic" if not args.triples_npz else "file",
                "config": {"workload": spec["name"], "V": V, "R": R, "E": E, "d": d, "B": B, "s": s,
                           "skewed": spec["skewed"], "dropout": "off (keep=1)", "relu": True,
                           "l2": "flushed between timed iterations (256 MB memset outside the event pair); inputs are "
                                 "%.0f MB per matrix" % (V_loc * d * 4 / 1e6),
                           "parallelism": ("%s x%d%s" % ("feature-shard (experimental)" if args.shard == "feature"
                                                         else "1d-node-shard (%s halo exchange, %s transport)" %
                                                         (args.halo, getattr(layer, "halo_transport", lambda: None)()
                                                          or "nccl"), world,
                                                         " of the same graph" if strong else " (graph grows with N)"))
                           if world > 1 else "single",
                           "messages": info[0], "block_algo": os.environ.get("RGCN_BLOCK_ALGO", "auto")},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
                "roofline_layer": roofline_layer, "cpu_baseline": cpu_baseline, "parity_check": parity,
                "stages_ms": stages, "graph_prep_ms": prep_ms, "wall_s_timed_region": wall1 - wall0}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
