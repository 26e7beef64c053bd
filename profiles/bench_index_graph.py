#!/usr/bin/env python3
"""Keyphrase graphs on an existing index on one GPU: east_graph_index_dev (tiles of documents scored into a bounded fp64
scratch, each tile read once by k_threshold_bytes to write one relevance-byte plane per threshold, then C = B B^T per
plane) against the device route a user had before it (east_score_table_dev into a documents x keyphrases table, then
east_cooc_dev), all on the same index.

Arms, device-timed with CUDA events on the call's stream, warmed up first, then alternated rep by rep:
  (a) east_graph_index_dev at one threshold (T = 1);
  (b) east_score_table_dev into a D x K fp64 device table + east_cooc_dev at that threshold;
  (c) east_graph_index_dev at T = 4 thresholds in one call;
  (d) four T = 1 calls of east_graph_index_dev, one per threshold.
Before timing, the counts of (a) and (b) and every plane of (c) and the matching call of (d) are compared element for
element.  A separate pass with option time_kernels = 1 gives the per-kernel split.

Collections:
  * headline: bench.py's collection (synth.packed_collection_fast(1000, 50 000), synth.keyphrases(1000)), one index;
  * configs[4]-shaped: 10^4 keyphrases x 10^5 documents x 10 KB in two device batches of 5 x 10^4, built once and
    reused; per rep every arm runs on both batches and the counts are summed on the device.

usage: python profiles/bench_index_graph.py [--out DIR] [--reps 10] [--config4-reps 5] [--warmup 2] [--kernel-reps 3]
Writes DIR/bench_index_graph_b200.json (default DIR: profiles/index_graph) and prints it."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "ast-text-analysis_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

THRESHOLD = 0.25                        # keyphrases_graph's default relevance threshold (-r)
THRESHOLDS = [0.15, 0.25, 0.35, 0.5]    # arm (c) / (d)
ARMS = ["a_graph_index_T1", "b_score_table_dev+cooc_dev", "c_graph_index_T4", "d_graph_index_4xT1"]


def _stats(ms):
    ms = sorted(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms[0]), "max_ms": float(ms[-1]), "reps": len(ms)}


def _alternate(arms, reps, warmup, stream):
    """{name: stats} of CUDA-event times around each arm, arms alternated rep by rep after `warmup` calls of each"""
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
    """{arm: {kernel: median ms per arm call}} with option time_kernels = 1, arms alternated"""
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
                got[name].setdefault(k, []).append((v["ms"], v["launches"]))
    return {name: {k: {"ms": float(np.median([m for m, _ in v])), "launches": int(np.median([n for _, n in v]))}
                   for k, v in ks.items()} for name, ks in got.items()}


def _shape_bytes(D, K, T):
    Dp, Kp = (D + 127) // 128 * 128, (K + 255) // 256 * 256
    return {"table_D_K_8": D * K * 8, "relevance_bytes_T_Kp_Dp": T * Kp * Dp, "T": T, "D": D, "K": K}


def _arms(torch, batches, codes, off, kp_dev, stream, K):
    """the four arms over `batches` [(DeviceIndex, D)], counts summed over the batches into device tensors"""
    from east import _capi
    dev = kp_dev.device
    T = len(THRESHOLDS)
    D_max = max(D for _, D in batches)
    S = torch.empty((D_max, K), dtype=torch.float64, device=dev)
    part = torch.empty((T, K, K), dtype=torch.int32, device=dev)
    out = {name: torch.zeros((T if name.startswith(("c_", "d_")) else 1, K, K), dtype=torch.int32, device=dev) for name in ARMS}
    s = stream.cuda_stream

    def graph(C, thresholds):
        C.zero_()
        for idx, D in batches:
            idx.graph_dev(kp_dev.data_ptr(), codes, off, thresholds, part.data_ptr(), stream=s)
            C.add_(part[:len(thresholds)].view_as(C))

    def a():
        graph(out["a_graph_index_T1"], [THRESHOLD])

    def b():
        C = out["b_score_table_dev+cooc_dev"]
        C.zero_()
        for idx, D in batches:
            idx.score_table_dev(kp_dev.data_ptr(), off, S.data_ptr(), stream=s)
            _capi.cooc_dev(S.data_ptr(), D, K, THRESHOLD, part.data_ptr(), stream=s)
            C.add_(part[0])

    def c():
        graph(out["c_graph_index_T4"], THRESHOLDS)

    def d():
        C = out["d_graph_index_4xT1"]
        C.zero_()
        for t, r in enumerate(THRESHOLDS):
            for idx, D in batches:
                idx.graph_dev(kp_dev.data_ptr(), codes, off, [r], part.data_ptr(), stream=s)
                C[t].add_(part[0])

    return [(ARMS[0], a), (ARMS[1], b), (ARMS[2], c), (ARMS[3], d)], out


def _check(torch, arms, out):
    for _, fn in arms:
        fn()
    torch.cuda.synchronize()
    t1 = THRESHOLDS.index(THRESHOLD)
    return {"a_equals_b": bool(torch.equal(out[ARMS[0]], out[ARMS[1]])),
            "c_equals_d_every_plane": bool(torch.equal(out[ARMS[2]], out[ARMS[3]])),
            "c_plane_of_0.25_equals_a": bool(torch.equal(out[ARMS[2]][t1], out[ARMS[0]][0]))}


def _section(torch, label, batches, codes, off, kp_dev, stream, K, reps, warmup, kernel_reps):
    arms, out = _arms(torch, batches, codes, off, kp_dev, stream, K)
    equal = _check(torch, arms, out)
    if not all(equal.values()):
        raise SystemExit("%s: the arms' counts differ: %r" % (label, equal))
    calls = _alternate(arms, reps, warmup, stream)
    kernels = _kernel_ms(arms, kernel_reps)
    D = sum(D for _, D in batches)
    med = {k: v["median_ms"] for k, v in calls.items()}
    return {
        "documents": D, "batches": len(batches), "keyphrases": K, "threshold_T1": THRESHOLD, "thresholds_T4": THRESHOLDS,
        "counts_equal": equal,
        "call_device_ms": calls,
        "ratios_of_medians": {"a_over_b": med[ARMS[0]] / med[ARMS[1]], "c_over_d": med[ARMS[2]] / med[ARMS[3]],
                              "c_over_a": med[ARMS[2]] / med[ARMS[0]]},
        "kernel_ms_median_per_arm_call": kernels,
        "score_bytes_by_shape_per_batch": [_shape_bytes(Db, K, T) for _, Db in batches for T in (1, len(THRESHOLDS))],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "index_graph"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--config4-reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-reps", type=int, default=3)
    ap.add_argument("--no-config4", action="store_true")
    args = ap.parse_args()

    import torch
    import synth
    from east import _capi, utils

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    res = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        res["nvidia_smi_name_power_limit_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        res["nvidia_smi_name_power_limit_max_sm_clock"] = "unavailable: %r" % (e,)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)

    # ---- headline collection: one index, device-resident keyphrases
    D, K = 1000, 1000
    text, doc_off, doc_m = synth.packed_collection_fast(D, 50000)
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(K)]
    codes, off = _capi.pack_keyphrases(prepared)
    text_dev = torch.from_numpy(text.view(np.int32)).to(dev)
    kp_dev = torch.from_numpy(codes.view(np.int32).copy()).to(dev)
    idx = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, stream=stream.cuda_stream)
    idx.wait()
    res["headline"] = _section(torch, "headline", [(idx, D)], codes, off, kp_dev, stream, K, args.reps, args.warmup,
                               args.kernel_reps)
    res["headline"]["what"] = ("synth.packed_collection_fast(1000, 50 000) indexed once (east_build_dev), synth.keyphrases(1000) "
                               "on the device, normalized scores")
    idx.close()
    del text_dev, kp_dev
    torch.cuda.empty_cache()
    _capi.trim(0)

    # ---- configs[4]-shaped: two device batches built once and reused
    if args.no_config4:
        res["config4"] = "not measured"
    else:
        K4, half = 10000, 50000
        prepared4 = [utils.prepare_text(k) for k in synth.keyphrases(K4)]
        c4, o4 = _capi.pack_keyphrases(prepared4)
        kp4 = torch.from_numpy(c4.view(np.int32).copy()).to(dev)
        batches, texts = [], []
        for b in range(2):
            t_b, off_b, m_b = synth.packed_collection_fast(half, 10000, first_seed=77 + b * 1000003)
            texts.append(torch.from_numpy(t_b.view(np.int32)).to(dev))
            ib = _capi.DeviceIndex.build_dev(texts[-1].data_ptr(), off_b, m_b, stream=stream.cuda_stream)
            ib.wait()
            batches.append((ib, half))
        res["config4"] = _section(torch, "config4", batches, c4, o4, kp4, stream, K4, args.config4_reps, 1, args.kernel_reps)
        res["config4"]["what"] = ("10^4 keyphrases x 10^5 documents x 10 KB (synth.packed_collection_fast), two device batches "
                                  "of 5 x 10^4 documents indexed once (east_build_dev); per rep every arm runs on both "
                                  "batches and sums the counts on the device")
        for ib, _ in batches:
            ib.close()

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_index_graph_b200.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
