#!/usr/bin/env python3
"""Synonym-expanded keyphrase table on one GPU: the grouped scoring call (east_score_groups_dev, k_score_combine_max)
against the plain table on the same index, and the per-variant path it replaces; the one-call synonym table
(east_table_groups_dev: the per-document kernel keeps the best variant of each group, k_doc_suffix_sort_groups) against
the plain one-call table and against build + grouped call; keyphrases_table with the synonimizer, one engine call from
str texts, against the previous route (host preprocessing and build, then the grouped call).

Workload: the headline collection of bench.py (synth.packed_collection_fast(1000, 50 000), synth.keyphrases(1000))
and synth.synonyms(): every keyphrase word gets 0-3 synonyms from the same Zipf, default_rng(11).

usage: python profiles/bench_synonyms.py [--out DIR] [--reps 20] [--warmup 3] [--sample-pairs 20] [--e2e-runs 3]
Writes DIR/bench_synonyms.json and prints it."""
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


def _stats(ms):
    ms = sorted(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": ms[0], "max_ms": ms[-1], "reps": len(ms)}


def _group_max(scores, group_off):
    out = np.empty(len(group_off) - 1, dtype=np.float64)
    for g in range(len(group_off) - 1):
        best = scores[group_off[g]]
        for v in range(group_off[g] + 1, group_off[g + 1]):
            if scores[v] > best:
                best = scores[v]
        out[g] = best
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_synonyms_out")
    ap.add_argument("--docs", type=int, default=1000)
    ap.add_argument("--doc-bytes", type=int, default=50000)
    ap.add_argument("--keyphrases", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample-pairs", type=int, default=20)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-runs", type=int, default=3)
    args = ap.parse_args()

    import torch
    import synth
    from east import _capi, applications, relevance, utils
    from east.asts.utils import codepoints
    from oracle import oracle

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    res = {"workload": {"docs": args.docs, "doc_bytes": args.doc_bytes, "keyphrases": args.keyphrases,
                        "synonyms": "synth.synonyms(seed=11): 0-3 Zipf synonyms per distinct keyphrase word"}}
    res["gpu"] = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        res["nvidia_smi_name_power_limit_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        res["nvidia_smi_name_power_limit_max_sm_clock"] = "unavailable: %r" % (e,)

    # ---- host: expansion + packing (timed), sizes
    prepared = [utils.prepare_text(k) for k in synth.keyphrases(args.keyphrases)]
    synonyms = synth.synonyms(prepared)
    t0 = time.perf_counter()
    vcodes, voff, group_off = _capi.pack_variant_groups(prepared, synonyms)
    res["host_expand_and_pack_ms"] = (time.perf_counter() - t0) * 1e3
    kcodes, koff = _capi.pack_keyphrases(prepared)
    V, G = len(voff) - 1, len(group_off) - 1

    def distinct_suffixes(codes, off):
        return len({codes[off[i] + s:off[i + 1]].tobytes() for i in range(len(off) - 1) for s in range(off[i + 1] - off[i])})

    res["sizes"] = {"keyphrases": G, "variants": V, "largest_group": int(np.diff(group_off).max()),
                    "suffixes_plain": int(koff[-1]), "suffixes_variants": int(voff[-1]),
                    "distinct_suffixes_plain": distinct_suffixes(kcodes, koff),
                    "distinct_suffixes_variants": distinct_suffixes(vcodes, voff)}

    # ---- device: one index, the grouped call and the plain table on it
    text, doc_off, doc_m = synth.packed_collection_fast(args.docs, args.doc_bytes)
    D = len(doc_m)
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    text_dev = torch.from_numpy(text.view(np.int32)).to(dev)
    vk_dev = torch.from_numpy(vcodes.view(np.int32).copy()).to(dev)
    kk_dev = torch.from_numpy(kcodes.view(np.int32).copy()).to(dev)
    out_g = torch.empty((D, G), dtype=torch.float64, device=dev)
    out_k = torch.empty((D, G), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    idx = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, stream=stream.cuda_stream)
    idx.wait()

    def grouped():
        idx.score_groups_dev(vk_dev.data_ptr(), voff, group_off, out_g.data_ptr(), stream=stream.cuda_stream)

    def plain():
        idx.score_table_dev(kk_dev.data_ptr(), koff, out_k.data_ptr(), True, stream=stream.cuda_stream)

    def timed(fn, name):
        # the first call prepares the keyphrases (kept for the next calls on this thread): host clock, the call syncs
        _capi.set_option("drop_kp_cache", 1)
        t = time.perf_counter()
        fn()
        first = (time.perf_counter() - t) * 1e3
        for _ in range(args.warmup):
            fn()
        ms = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.reps):
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        out = _stats(ms)
        out["first_call_with_preparation_host_ms"] = first
        res[name] = out

    timed(grouped, "device_ms_score_groups_dev")
    timed(plain, "device_ms_score_table_dev_plain_keyphrases")

    # ---- one engine call: build + score, alternated; each call builds (and frees) its own index
    out_1 = torch.empty((D, G), dtype=torch.float64, device=dev)

    def one_call_groups():
        _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, vk_dev.data_ptr(), vcodes, voff, out_1.data_ptr(),
                                              stream=stream.cuda_stream, group_off=group_off).close()

    def one_call_plain():
        _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kk_dev.data_ptr(), kcodes, koff, out_k.data_ptr(),
                                              True, stream=stream.cuda_stream).close()

    def build_then_groups():
        i2 = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, stream=stream.cuda_stream)
        i2.score_groups_dev(vk_dev.data_ptr(), voff, group_off, out_g.data_ptr(), stream=stream.cuda_stream)
        i2.close()

    def one_call_groups_batched():
        _capi.set_option("no_fused_score", 1)
        try:
            one_call_groups()
        finally:
            _capi.set_option("no_fused_score", 0)

    arms = (("east_table_groups_dev", one_call_groups), ("east_table_groups_dev_no_fused_score", one_call_groups_batched),
            ("east_table_dev_plain", one_call_plain), ("east_build_dev_then_east_score_groups_dev", build_then_groups))
    for _, fn in arms:
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    per_arm = {name: [] for name, _ in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.reps):
        for name, fn in arms:
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            per_arm[name].append(e0.elapsed_time(e1))
    res["one_call_device_ms"] = {name: _stats(ms) for name, ms in per_arm.items()}
    res["one_call_note"] = ("CUDA events on the call's stream around the whole call (build, scoring, index freed), arms "
                            "alternated rep by rep; text, keyphrases and table device-resident; no_fused_score = the per-run "
                            "batched scorer (k_score_suffixes + k_score_combine_max) after the per-document kernel")
    one = res["one_call_device_ms"]
    res["one_call_groups_over_plain"] = one["east_table_groups_dev"]["median_ms"] / one["east_table_dev_plain"]["median_ms"]
    res["one_call_groups_over_no_fused_score"] = (one["east_table_groups_dev"]["median_ms"] /
                                                  one["east_table_groups_dev_no_fused_score"]["median_ms"])
    res["one_call_groups_over_build_then_groups"] = (one["east_table_groups_dev"]["median_ms"] /
                                                     one["east_build_dev_then_east_score_groups_dev"]["median_ms"])
    res["device_note"] = ("CUDA events on the call's stream, preparation cached (same keyphrases as the previous call); the "
                          "per-suffix scratch (documents x distinct suffixes doubles) exceeds the 126 MB L2")
    res["grouped_over_plain"] = (res["device_ms_score_groups_dev"]["median_ms"] /
                                 res["device_ms_score_table_dev_plain_keyphrases"]["median_ms"])

    # ---- per-kernel split (separate short pass: an event pair around every launch)
    split = {}
    for name, fn in (("score_groups_dev", grouped), ("score_table_dev_plain", plain)) + arms:
        fn()
        _capi.set_option("time_kernels", 0)
        _capi.set_option("time_kernels", 1)
        for _ in range(3):
            fn()
        ks = _capi.kernel_stats()
        _capi.set_option("time_kernels", 0)
        split[name] = {k: {"ms_per_call": v["ms"] / 3, "launches_per_call": v["launches"] / 3} for k, v in ks.items()}
    res["kernel_split"] = split

    # ---- the old path: one east_score_one per variant per (text, keyphrase) pair, on a fixed sample of pairs
    rng = np.random.default_rng(5)
    pairs = [(int(rng.integers(0, D)), int(rng.integers(0, G))) for _ in range(args.sample_pairs)]
    idx.score_one(0, codepoints("A"))
    t = time.perf_counter()
    old = []
    for d, k in pairs:
        old.append(max(idx.score_one(d, codepoints(v)) for v in utils.synonym_variants(prepared[k], synonyms)))
    per_pair = (time.perf_counter() - t) / len(pairs)
    res["old_path_per_variant_score_one"] = {
        "sampled_pairs": len(pairs), "host_ms_per_pair": per_pair * 1e3,
        "extrapolated_table_s": per_pair * D * G,
        "note": "EXTRAPOLATION: host wall time of the sampled pairs x documents x keyphrases, not a measured table"}

    # ---- parity, after the timed region: sampled rows against the oracle's max over each group
    grouped()
    plain()
    one_call_groups()
    torch.cuda.synchronize()
    table = out_g.cpu().numpy()
    plain_table = out_k.cpu().numpy()
    one_call_table = out_1.cpu().numpy()
    checked, ok = [], True
    for d in sorted({0, D // 2, D - 1}):
        o = oracle.OracleEASA(text=text[doc_off[d]:doc_off[d + 1]], m=int(doc_m[d]))
        exp = _group_max(o.score_many(vcodes, voff, True), group_off)
        ok &= bool(np.array_equal(table[d].view(np.uint64), exp.view(np.uint64)))
        ok &= bool(np.array_equal(plain_table[d].view(np.uint64), o.score_many(kcodes, koff, True).view(np.uint64)))
        checked.append(d)
    for (d, k), v in zip(pairs, old):
        ok &= float(v) == float(table[d, k])
    ok &= bool(np.array_equal(one_call_table.view(np.uint64), table.view(np.uint64)))   # every row
    res["parity"] = {"rows_checked_against_oracle": checked, "old_path_pairs_checked": len(pairs),
                     "one_call_table_rows_checked_against_grouped_call": D, "bit_exact": ok}
    res["grouped_at_least_plain"] = bool((table >= plain_table).all())

    # ---- end to end: applications.keyphrases_table with the synonimizer from str texts.  New: one engine call per
    # device batch (device preprocessing, build, in-kernel groups).  Old route: set_text_collection without the
    # keyphrases (host preprocessing, build), then relevance_table's grouped call.  Alternated run by run.
    if not args.no_e2e:
        class Synonimizer(object):
            def get_synonyms(self):
                return synonyms

        phases = {"set_text_collection_s": [], "relevance_table_s": []}

        class OldRoute(relevance.ASTRelevanceMeasure):
            def set_text_collection(self, texts, language=None, prepared_keyphrases=None, synonimizer=None):
                t = time.perf_counter()
                super(OldRoute, self).set_text_collection(texts, language)
                phases["set_text_collection_s"].append(time.perf_counter() - t)

            def relevance_table(self, prepared_keyphrases, synonimizer=None):
                t = time.perf_counter()
                out = super(OldRoute, self).relevance_table(prepared_keyphrases, synonimizer)
                phases["relevance_table_s"].append(time.perf_counter() - t)
                return out

        texts = {"t%d" % j: d for j, d in enumerate(synth.documents(args.docs, args.doc_bytes))}
        kps = synth.keyphrases(args.keyphrases)
        grouped_calls = []
        real_score_groups = _capi.DeviceIndex.score_groups

        def counting(self, *a, **k):
            grouped_calls.append(1)
            return real_score_groups(self, *a, **k)
        _capi.DeviceIndex.score_groups = counting
        walls = {"new": [], "old_route": []}
        tabs = {}
        new_one_call = True
        for _ in range(args.e2e_runs):
            for name, make in (("new", relevance.ASTRelevanceMeasure), ("old_route", OldRoute)):
                measure = make()
                del grouped_calls[:]
                t = time.perf_counter()
                tabs[name] = applications.keyphrases_table(kps, texts, measure, synonimizer=Synonimizer())
                walls[name].append(time.perf_counter() - t)
                if name == "new":   # device preprocessing, one batch, no grouped call after the build
                    new_one_call &= (measure.asts[0]._strings_collection is None and len(measure._batches) == 1
                                     and not grouped_calls)
                del measure
        _capi.DeviceIndex.score_groups = real_score_groups
        res["e2e_keyphrases_table_with_synonimizer_s"] = {
            "new": {"runs_s": walls["new"], "median_s": float(np.median(walls["new"]))},
            "old_route": {"runs_s": walls["old_route"], "median_s": float(np.median(walls["old_route"])),
                          "phases": phases},
            "old_over_new": float(np.median(walls["old_route"]) / np.median(walls["new"])),
            "new_is_one_engine_call_with_device_preprocessing": bool(new_one_call),
            "note": "host wall time of applications.keyphrases_table, synth.documents(%d, %d) as str, dict building included; "
                    "runs alternated, run 1 of each arm is cold; old_route phases: set_text_collection(texts) (host "
                    "preprocessing + build) and relevance_table(prepared, synonimizer) (grouped call)"
                    % (args.docs, args.doc_bytes)}
        tab = tabs["new"]
        res["parity"]["e2e_new_equals_old_route"] = all(
            float(tabs["new"][kp][n]).hex() == float(tabs["old_route"][kp][n]).hex() for kp in kps for n in texts)
        name = "t0"
        o = oracle.OracleEASA(utils.text_to_strings_collection(texts[name]))
        exp = _group_max(o.score_many(vcodes, voff, True), group_off)
        got = np.array([tab[kp][name] for kp in kps], dtype=np.float64)
        res["parity"]["e2e_text_t0_bit_exact"] = bool(np.array_equal(got.view(np.uint64), exp.view(np.uint64)))

    idx.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_synonyms.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
