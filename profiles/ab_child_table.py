#!/usr/bin/env python3
"""A/B of phase 8 of the per-document kernel: tiles of 32 ranks (the default) against the per-thread stack walk
(EAST_DOC_SORT_STACK_WALK=1).  The switch is read once per process, so every arm is a process of its own, on the same
build, alternated: `bench.py` (ms_per_step of the device-timed step and the k_doc_suffix_sort event time per step), then
one profiled call per arm (EAST_DOC_SORT_PROFILE=1: SM cycles per phase and document, the tile path's query counts).
usage (GPU box): python profiles/ab_child_table.py [--rounds 3] [--steps 30] [--warmup 5]"""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROFILED_CALL = """
import sys, os
sys.path.insert(0, os.path.join(%r, "ast-text-analysis_b200")); sys.path.insert(0, %r)
import numpy as np, torch
import synth
from east import _capi, utils
packed, ms, _ = synth.packed_collection(1000, 50000)
doc_off = np.zeros(1001, dtype=np.int64); np.cumsum([len(p) for p in packed], out=doc_off[1:])
dev = torch.from_numpy(np.concatenate(packed).view(np.int32)).cuda()
codes, off = _capi.pack_keyphrases([utils.prepare_text(k) for k in synth.keyphrases(1000)])
kp_dev = torch.from_numpy(codes.view(np.int32).copy()).cuda()
out_dev = torch.empty(1000 * 1000, dtype=torch.float64, device="cuda")
for _ in range(2):
    _capi.DeviceIndex.build_dev_and_score(dev.data_ptr(), doc_off, np.array(ms, dtype=np.int32), kp_dev.data_ptr(), codes, off,
                                          out_dev.data_ptr(), True).close()
torch.cuda.synchronize()
""" % (ROOT, ROOT)


def env_for(arm, **extra):
    env = dict(os.environ)
    env.pop("EAST_DOC_SORT_STACK_WALK", None)
    if arm == "stack_walk":
        env["EAST_DOC_SORT_STACK_WALK"] = "1"
    env.update(extra)
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    print(json.dumps({"gpu": smi.stdout.strip()}), flush=True)
    for r in range(a.rounds):
        for arm in ("tiles", "stack_walk"):
            cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(a.steps), "--warmup",
                   str(a.warmup), "--no-extras", "--no-cpu-baseline"]
            res = subprocess.run(cmd, env=env_for(arm), cwd=ROOT, capture_output=True, text=True)
            line = next((json.loads(x) for x in reversed(res.stdout.splitlines()) if x.startswith("{")), None)
            if line is None:
                print(res.stdout[-2000:], res.stderr[-4000:], flush=True)
                raise SystemExit("bench.py gave no result line (%s)" % arm)
            k = line.get("breakdown", {}).get("kernels", {}).get("k_doc_suffix_sort") or {}
            print(json.dumps({"round": r, "arm": arm, "ms_per_step": line["ms_per_step"],
                              "k_doc_suffix_sort_ms_per_step": k.get("ms_per_step"),
                              "e2e_ms_per_step": line.get("e2e", {}).get("ms_per_step"),
                              "parity_checked": line.get("parity_checked")}), flush=True)
    for arm in ("tiles", "stack_walk"):
        res = subprocess.run([sys.executable, "-c", PROFILED_CALL], env=env_for(arm, EAST_DOC_SORT_PROFILE="1"), cwd=ROOT,
                             capture_output=True, text=True)
        lines = [x for x in res.stderr.splitlines() if x.startswith("[east] doc_sort")]
        print(json.dumps({"arm": arm, "profile": lines[-2:], "rc": res.returncode}), flush=True)
        if res.returncode:
            print(res.stderr[-4000:], flush=True)


if __name__ == "__main__":
    main()
