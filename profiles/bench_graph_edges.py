#!/usr/bin/env python3
"""Keyphrase graphs assembled on the device (east_graph_edges_dev / _host, applications.graph_on_device) against the host
assembly they replace (applications.graph_from_cooccurrence: numpy over all K^2 cells after the counts were copied to the
host), on one GPU.

Sections:
  * config4: counts of a configs[4]-shaped graph call -- 10^4 keyphrases x 10^5 documents x 10 KB
    (synth.packed_collection_fast) in two device batches of 5 x 10^4, east_graph_index_dev at r = 0.25 summed on the
    device.  On the same device counts, at (c, p) = (0.6, 1) -- or, when c = 0.6 gives more than 2 x 10^6 edges, at the
    first of c = 0.8, 0.9, 0.95, 0.99, 1.0 that gives fewer (the JSON records the edges at each c it tried):
      - per-kernel device time of the assembly (option time_kernels = 1): k_graph_supports, k_graph_edge_count,
        k_graph_edge_emit;
      - host wall time of the whole east_graph_edges_dev call (it returns with the edges on the host), of
        graph_on_device (the call plus the graph dict), and of the route it replaces: the K x K copy to the host plus
        graph_from_cooccurrence.  Alternated rep by rep after a warm-up.
    Both dicts are compared (confidences by float.hex) before timing.
  * k30k (unless --no-k30k): the device side at 3 x 10^4 keyphrases on the same index; the host route is not run there
    (it needs a 3.6 GB copy and 7.2 GB of float64 on the host).
  * public: applications.keyphrases_graph wall time on 1000 raw texts x 50 KB (the headline collection's size; device
    preprocessing) with 10^4 keyphrases, (c, r, p) = (0.6, 0.25, 1), c chosen as above: "after" as it stands, "before" with the graph
    assembled by graph_from_cooccurrence as at the parent commit; alternated, graphs compared.

usage: python profiles/bench_graph_edges.py [--out DIR] [--reps 5] [--public-reps 3] [--no-config4] [--no-k30k]
Writes DIR/bench_graph_edges_b200.json (default DIR: profiles/graph_edges) and prints it."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "ast-text-analysis_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

C_CONF, R_THR, P_SUP = 0.6, 0.25, 1
C_SPARSER = [0.8, 0.9, 0.95, 0.99, 1.0]   # when c = 0.6 gives more edges than a graph dict can hold in reasonable time
MAX_DICT_EDGES = 2000000


def _log(*a):
    print(*a, flush=True)


def _edge_count(C, node_col, c):
    """edges of all planes of the counts C (numpy or CUDA tensor) at referral confidence c: a sizing call, edge_cap = 0"""
    import ctypes
    from east import _capi
    L = _capi.load()
    i32, i64 = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
    N = len(node_col)
    support, n_edges = np.empty(N, np.int32), np.zeros(1, np.int64)
    rc = L.east_graph_edges_dev(ctypes.c_void_p(C.data_ptr()), C.shape[-1], 1, node_col.ctypes.data_as(i32), N, c, P_SUP,
                                C.device.index, None, support.ctypes.data_as(i32), n_edges.ctypes.data_as(i64), 0, None, None, None)
    assert rc in (0, _capi.EAST_ERR_RANGE), rc
    return int(n_edges[0])


def _referral_confidence(C, node_col):
    """(c, {c: edges}): C_CONF, or the first of C_SPARSER whose graph has at most MAX_DICT_EDGES edges"""
    seen = {}
    for c in [C_CONF] + C_SPARSER:
        seen[c] = _edge_count(C, node_col, c)
        if seen[c] <= MAX_DICT_EDGES:
            return c, seen
    return c, seen


def _stats(ms):
    ms = sorted(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms[0]), "max_ms": float(ms[-1]), "reps": len(ms)}


def _wall(fn):
    t = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t) * 1e3, out


def _key(graph):
    return (graph["nodes"], [(e["source"], e["target"], float(e["confidence"]).hex()) for e in graph["edges"]])


def _counts(torch, batches, codes, off, kp_dev, K, stream):
    """int32 [K, K] counts of the index batches at R_THR, summed on the device"""
    C = torch.zeros((K, K), dtype=torch.int32, device=kp_dev.device)
    part = torch.empty_like(C)
    for idx in batches:
        idx.graph_dev(kp_dev.data_ptr(), codes, off, R_THR, part.data_ptr(), stream=stream.cuda_stream)
        C += part
    torch.cuda.synchronize()
    return C


def _section(torch, C_dev, K, reps, host_reps):
    """host_reps = 0: the host route is not run (at 3 x 10^4 keyphrases it needs a 3.6 GB copy and 7.2 GB of float64)"""
    from east import _capi, applications
    kps = ["kp%d" % k for k in range(K)]   # one node per column
    node_col = np.arange(K, dtype=np.int32)
    c_used, edges_at = _referral_confidence(C_dev, node_col)
    _log("K = %d: edges per referral confidence %r, timing c = %r" % (K, edges_at, c_used))

    def call():
        return _capi.graph_edges(C_dev, node_col, c_used, P_SUP)

    def device():
        return applications.graph_on_device(kps, kps, C_dev, c_used, R_THR, P_SUP)

    def host():
        return applications.graph_from_cooccurrence(kps, kps, C_dev.cpu().numpy(), c_used, R_THR, P_SUP)

    dev_graph = device()
    equal = "not measured"
    times = {"east_graph_edges_dev_call": [], "graph_on_device": []}
    if host_reps:
        ms_host, host_graph = _wall(host)
        equal = _key(dev_graph) == _key(host_graph)
        if not equal:
            raise SystemExit("K = %d: the device graph differs from graph_from_cooccurrence" % K)
        times["copy_KxK_to_host+graph_from_cooccurrence"] = [ms_host]
    call()
    for rep in range(reps):
        times["east_graph_edges_dev_call"].append(_wall(call)[0])
        times["graph_on_device"].append(_wall(device)[0])
        if rep + 1 < host_reps:
            times["copy_KxK_to_host+graph_from_cooccurrence"].append(_wall(host)[0])
    copy = [_wall(lambda: C_dev.cpu())[0] for _ in range(3)]
    kernels = {}
    for _ in range(3):
        _capi.set_option("time_kernels", 0)
        _capi.set_option("time_kernels", 1)
        try:
            call()
            for k, v in _capi.kernel_stats().items():
                kernels.setdefault(k, []).append((v["ms"], v["launches"], v["bytes"]))
        finally:
            _capi.set_option("time_kernels", 0)
    kernel_ms = {k: {"ms": float(np.median([m for m, _, _ in v])), "launches": int(v[0][1]), "algorithmic_bytes": v[0][2],
                     "GB_per_s": v[0][2] / (np.median([m for m, _, _ in v]) * 1e6)} for k, v in kernels.items()}
    med = {k: _stats(v)["median_ms"] for k, v in times.items()}
    return {
        "keyphrases": K, "c": c_used, "r": R_THR, "p": P_SUP, "edges_per_referral_confidence": {repr(k): v for k, v in edges_at.items()},
        "nodes": len(dev_graph["nodes"]), "edges": len(dev_graph["edges"]), "graphs_equal_hex": equal,
        "wall_ms": {k: _stats(v) for k, v in times.items()},
        "copy_KxK_to_host_ms": _stats(copy),
        "kernel_ms_median_per_call": kernel_ms,
        "host_route_over_graph_on_device": (med["copy_KxK_to_host+graph_from_cooccurrence"] / med["graph_on_device"]
                                            if host_reps else "not measured"),
    }


def _public(reps):
    """keyphrases_graph after (device assembly) and before (graph_from_cooccurrence), alternated"""
    import synth
    from east import applications, relevance
    texts = {"t%d" % i: d for i, d in enumerate(synth.documents(1000, 50000, first_seed=4242))}
    kps = synth.keyphrases(10000, seed=11)
    device_assembly = applications.graph_on_device
    counts = {}

    def before_assembly(keyphrases, kept, cooc, c, r, p):
        return applications.graph_from_cooccurrence(keyphrases, kept, cooc, c, r, p)

    def sizing(keyphrases, kept, cooc, c, r, p):
        counts["cooc"], counts["node_col"] = cooc, applications._node_columns(keyphrases, kept)
        return {"nodes": [], "edges": []}

    def run(assembly, c):
        applications.graph_on_device = assembly
        try:
            return applications.keyphrases_graph(kps, texts, c, R_THR, P_SUP, similarity_measure=relevance.ASTRelevanceMeasure())
        finally:
            applications.graph_on_device = device_assembly

    import torch
    run(sizing, C_CONF)
    c_used, edges_at = _referral_confidence(torch.from_numpy(counts["cooc"]).cuda(), counts["node_col"])
    _log("public: edges per referral confidence %r, timing c = %r" % (edges_at, c_used))
    after, before = run(device_assembly, c_used), run(before_assembly, c_used)   # warm-up
    equal = _key(after) == _key(before)
    if not equal:
        raise SystemExit("keyphrases_graph: the device graph differs from the host graph")
    times = {"after": [], "before": []}
    for _ in range(reps):
        times["after"].append(_wall(lambda: run(device_assembly, c_used))[0])
        times["before"].append(_wall(lambda: run(before_assembly, c_used))[0])
        _log("public: after %.1f ms, before %.1f ms" % (times["after"][-1], times["before"][-1]))
    med = {k: _stats(v)["median_ms"] for k, v in times.items()}
    return {"what": "applications.keyphrases_graph(synth.keyphrases(10^4), 1000 raw texts x 50 KB (synth.documents), c, 0.25, 1), "
                    "default ASTRelevanceMeasure; before = graph_from_cooccurrence on the host counts (the parent's route)",
            "c": c_used, "edges_per_referral_confidence": {repr(k): v for k, v in edges_at.items()},
            "nodes": len(after["nodes"]), "edges": len(after["edges"]), "graphs_equal_hex": equal,
            "wall_ms": {k: _stats(v) for k, v in times.items()}, "before_over_after": med["before"] / med["after"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "graph_edges"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--public-reps", type=int, default=3)
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--no-k30k", action="store_true")
    args = ap.parse_args()

    import torch
    import synth
    from east import _capi, utils

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    res = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        res["nvidia_smi_name_power_limit_sm_clock_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        res["nvidia_smi_name_power_limit_sm_clock_max_sm_clock"] = "unavailable: %r" % (e,)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)

    res["public"] = _public(args.public_reps)
    _log("public done")

    if args.no_config4:
        res["config4"] = res["k30k"] = "not measured"
    else:
        half = 50000
        batches, texts = [], []
        for b in range(2):
            t_b, off_b, m_b = synth.packed_collection_fast(half, 10000, first_seed=77 + b * 1000003)
            _log("config4: batch %d generated" % b)
            texts.append(torch.from_numpy(t_b.view(np.int32)).to(dev))
            ib = _capi.DeviceIndex.build_dev(texts[-1].data_ptr(), off_b, m_b, stream=stream.cuda_stream)
            ib.wait()
            batches.append(ib)
        for label, K, host_reps in (("config4", 10000, args.reps), ("k30k", 30000, 0)):
            if label == "k30k" and args.no_k30k:
                res[label] = "not measured"
                continue
            prepared = [utils.prepare_text(k) for k in synth.keyphrases(K)]
            codes, off = _capi.pack_keyphrases(prepared)
            kp_dev = torch.from_numpy(codes.view(np.int32).copy()).to(dev)
            C_dev = _counts(torch, batches, codes, off, kp_dev, K, stream)
            res[label] = _section(torch, C_dev, K, args.reps, host_reps)
            _log("%s done" % label)
            res[label]["what"] = ("counts of synth.keyphrases(%d) x 10^5 documents x 10 KB (synth.packed_collection_fast, two "
                                  "device batches, east_graph_index_dev at r = 0.25, summed on the device)" % K)
            del C_dev, kp_dev
            torch.cuda.empty_cache()
        for ib in batches:
            ib.close()

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_graph_edges_b200.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
