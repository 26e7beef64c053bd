#!/usr/bin/env python3
"""Keyphrase graphs without the score table on one GPU: east_graph_dev (the per-document kernel writes the relevance bytes
of C = B B^T, k_doc_suffix_sort_graph / k_doc_suffix_sort_groups_graph) against the table route it replaces
(east_table_dev, then east_cooc_dev: fp64 table, k_threshold_bytes, the same GEMM).

Sections (arms alternated rep by rep, medians with min / max):
  * benchmark collection (bench.py's headline: synth.packed_collection_fast(1000, 50 000), synth.keyphrases(1000)),
    device-resident, plain and with the seeded dictionary of synth.synonyms: whole calls (CUDA events on the call's
    stream) and the per-kernel times of the scoring kernels (option time_kernels);
  * the public API: applications.keyphrases_graph from str texts against the table route reproduced here
    (applications._score_matrix + _capi.cooc_host + graph_from_cooccurrence), host wall clock;
  * BASELINE configs[4] (10^4 keyphrases x 10^5 documents x 10 KB) on one GPU in two device batches, device-resident,
    batch by batch: east_graph_dev + a device-side sum of the counts against east_table_dev + east_cooc_dev, and the
    bytes each route allocates for scores (D K 8 against Kp Dp).
Every arm's counts are compared element for element with the other route's.

usage: python profiles/bench_graph.py [--out DIR] [--reps 10] [--warmup 2] [--e2e-runs 3] [--config4-reps 3] [--no-config4]
Writes DIR/bench_graph.json and prints it."""
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

THRESHOLD = 0.25   # keyphrases_graph's default relevance threshold (-r)


def _stats(ms):
    ms = sorted(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms[0]), "max_ms": float(ms[-1]), "reps": len(ms)}


def _alternate(arms, reps, warmup, stream):
    """{name: stats} of CUDA-event times around each arm's whole call, arms alternated rep by rep"""
    import torch
    for _, fn in arms:
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    per_arm = {name: [] for name, _ in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        for name, fn in arms:
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            per_arm[name].append(e0.elapsed_time(e1))
    return {name: _stats(ms) for name, ms in per_arm.items()}


def _kernel_ms(arms, reps):
    """{arm: {kernel: median ms per call}} with option time_kernels, arms alternated"""
    from east import _capi
    got = {name: {} for name, _ in arms}
    for _ in range(reps):
        for name, fn in arms:
            _capi.set_option("time_kernels", 0)
            _capi.set_option("time_kernels", 1)
            try:
                fn()
                stats = _capi.kernel_stats()
            finally:
                _capi.set_option("time_kernels", 0)
            for k, v in stats.items():
                got[name].setdefault(k, []).append(v["ms"])
    return {name: {k: float(np.median(v)) for k, v in ks.items()} for name, ks in got.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_graph_out")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-reps", type=int, default=5)
    ap.add_argument("--e2e-runs", type=int, default=3)
    ap.add_argument("--config4-reps", type=int, default=3)
    ap.add_argument("--no-config4", action="store_true")
    args = ap.parse_args()

    import torch
    import synth
    from east import _capi, applications, relevance, utils

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    res = {"threshold": THRESHOLD, "gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        res["nvidia_smi_name_power_limit_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        res["nvidia_smi_name_power_limit_max_sm_clock"] = "unavailable: %r" % (e,)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)

    # ---- benchmark collection, device-resident
    D, K = 1000, 1000
    text, doc_off, doc_m = synth.packed_collection_fast(D, 50000)
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(K)]
    kcodes, koff = _capi.pack_keyphrases(prepared)
    vcodes, voff, group_off = _capi.pack_variant_groups(prepared, synth.synonyms(prepared))
    res["benchmark_collection"] = {"docs": D, "doc_bytes": 50000, "code_points": int(doc_off[-1]), "keyphrases": K,
                                   "variants": len(voff) - 1}
    text_dev = torch.from_numpy(text.view(np.int32)).to(dev)
    kk_dev = torch.from_numpy(kcodes.view(np.int32).copy()).to(dev)
    vk_dev = torch.from_numpy(vcodes.view(np.int32).copy()).to(dev)
    S = torch.empty((D, K), dtype=torch.float64, device=dev)
    C_table = torch.empty((K, K), dtype=torch.int32, device=dev)
    C_graph = torch.empty((K, K), dtype=torch.int32, device=dev)

    def arms_for(codes, off, kp_dev, groups):
        def graph():
            _capi.DeviceIndex.build_dev_and_graph(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), codes, off, THRESHOLD,
                                                  C_graph.data_ptr(), True, stream=stream.cuda_stream, group_off=groups).close()

        def table():
            _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), codes, off, S.data_ptr(),
                                                  True, stream=stream.cuda_stream, group_off=groups).close()
            _capi.cooc_dev(S.data_ptr(), D, K, THRESHOLD, C_table.data_ptr(), stream=stream.cuda_stream)
        return [("east_graph_dev", graph), ("east_table_dev+east_cooc_dev", table)]

    for label, (codes, off, kp_dev, groups) in (("plain", (kcodes, koff, kk_dev, None)),
                                                ("synonyms", (vcodes, voff, vk_dev, group_off))):
        arms = arms_for(codes, off, kp_dev, groups)
        calls = _alternate(arms, args.reps, args.warmup, stream)
        torch.cuda.synchronize()
        equal = bool(torch.equal(C_graph, C_table))
        kernels = _kernel_ms(arms, args.kernel_reps)
        scorer = "k_doc_suffix_sort_groups" if groups is not None else "k_doc_suffix_sort"
        res["benchmark_" + label] = {
            "call_device_ms": calls,
            "graph_over_table_route": calls["east_graph_dev"]["median_ms"] / calls["east_table_dev+east_cooc_dev"]["median_ms"],
            "counts_equal": equal,
            "kernel_ms_median": kernels,
            "scoring_kernel_ms": {scorer + "_graph": kernels["east_graph_dev"].get(scorer + "_graph"),
                                  scorer: kernels["east_table_dev+east_cooc_dev"].get(scorer)},
        }
    del S, C_table, C_graph, text_dev
    torch.cuda.empty_cache()
    _capi.trim(0)

    # ---- public API from str texts (host wall clock; the calls end on a synchronise)
    texts = {"t%d" % j: t for j, t in enumerate(synth.documents(D, 50000, first_seed=4242))}
    kps = synth.keyphrases(K)

    def api_graph():
        return applications.keyphrases_graph(kps, texts, similarity_measure=relevance.ASTRelevanceMeasure())

    def api_table_route():
        kept, _, scores = applications._score_matrix(kps, texts, relevance.ASTRelevanceMeasure(), None, "english")
        return applications.graph_from_cooccurrence(kps, kept, _capi.cooc_host(scores, THRESHOLD), 0.6, THRESHOLD, 1)

    walls = {"keyphrases_graph": [], "table_route": []}
    graphs = {}
    api_graph()
    for _ in range(args.e2e_runs):
        for name, fn in (("keyphrases_graph", api_graph), ("table_route", api_table_route)):
            t0 = time.perf_counter()
            graphs[name] = fn()
            walls[name].append((time.perf_counter() - t0) * 1e3)
    res["public_api_from_str_texts"] = {
        "what": "applications.keyphrases_graph(synth.keyphrases(1000), 1000 str texts of 50 KB) against "
                "_score_matrix + cooc_host + graph_from_cooccurrence, host wall clock, alternated, after one warm-up call",
        "wall_ms": {k: _stats(v) for k, v in walls.items()},
        "graphs_equal": graphs["keyphrases_graph"] == graphs["table_route"]}
    del texts
    _capi.trim(0)

    # ---- BASELINE configs[4] on one GPU: two device batches, batch by batch
    if args.no_config4:
        res["config4"] = "not measured"
    else:
        K4, D4, half = 10000, 100000, 50000
        prepared4 = [utils.prepare_text(k) for k in synth.keyphrases(K4)]
        c4, o4 = _capi.pack_keyphrases(prepared4)
        kp4 = torch.from_numpy(c4.view(np.int32).copy()).to(dev)
        batches = []
        for b in range(2):
            t_b, off_b, m_b = synth.packed_collection_fast(half, 10000, first_seed=77 + b * 1000003)
            batches.append((torch.from_numpy(t_b.view(np.int32)).to(dev), off_b, m_b))
        S4 = torch.empty((half, K4), dtype=torch.float64, device=dev)
        C_sum_g = torch.zeros((K4, K4), dtype=torch.int32, device=dev)
        C_sum_t = torch.zeros((K4, K4), dtype=torch.int32, device=dev)
        C_part = torch.empty((K4, K4), dtype=torch.int32, device=dev)

        def graph4():
            C_sum_g.zero_()
            for t_d, off_b, m_b in batches:
                _capi.DeviceIndex.build_dev_and_graph(t_d.data_ptr(), off_b, m_b, kp4.data_ptr(), c4, o4, THRESHOLD, C_part.data_ptr(),
                                                      True, stream=stream.cuda_stream).close()
                C_sum_g.add_(C_part)

        def table4():
            C_sum_t.zero_()
            for t_d, off_b, m_b in batches:
                _capi.DeviceIndex.build_dev_and_score(t_d.data_ptr(), off_b, m_b, kp4.data_ptr(), c4, o4, S4.data_ptr(), True,
                                                      stream=stream.cuda_stream).close()
                _capi.cooc_dev(S4.data_ptr(), half, K4, THRESHOLD, C_part.data_ptr(), stream=stream.cuda_stream)
                C_sum_t.add_(C_part)

        calls = _alternate([("east_graph_dev", graph4), ("east_table_dev+east_cooc_dev", table4)], args.config4_reps, 1, stream)
        torch.cuda.synchronize()
        Dp = (half + 127) // 128 * 128
        Kp = (K4 + 255) // 256 * 256
        res["config4"] = {
            "what": "10^4 keyphrases x 10^5 documents x 10 KB (synth.packed_collection_fast), two device batches of 5 x 10^4 "
                    "documents, device-resident; per rep both batches and a device-side sum of the counts",
            "code_points": int(sum(int(b[1][-1]) for b in batches)),
            "call_device_ms": calls,
            "graph_over_table_route": calls["east_graph_dev"]["median_ms"] / calls["east_table_dev+east_cooc_dev"]["median_ms"],
            "counts_equal": bool(torch.equal(C_sum_g, C_sum_t)),
            "score_bytes_per_batch": {"table_route_D_K_8": half * K4 * 8, "graph_Kp_Dp": Kp * Dp},
            "score_bytes_whole_collection_one_batch": {"table_route_D_K_8": D4 * K4 * 8,
                                                       "graph_Kp_Dp": Kp * ((D4 + 127) // 128 * 128)}}

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_graph.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
