#!/usr/bin/env python3
"""bench.py -- headline benchmark of the EASA hot path on B200.

Metric (BASELINE.json): AST keyphrase x document scores per second.  One "step" is one pass of the
whole hot path over one batch of synthetic documents: build the annotated suffix structure of every
document (suffix array, LCP, child table, annotation) and score every keyphrase against every
document -- i.e. what east.applications.keyphrases_table does (applications.py:11-56).

Workload at N=1: BASELINE.json configs[1]: 1 000 keyphrases x 1 000 synthetic Zipf documents of
~50 KB (SURVEY 8(d) generator, synth.py).  N>1: weak scaling, every rank indexes and scores its own
1 000 documents against the same 1 000 keyphrases and the per-rank [D_r, K] fp64 score slices are
joined with one NCCL all-gather inside the timed step.

  value      device-timed (CUDA events), inputs resident in HBM, max over ranks
  e2e        same step through the host-buffer C-ABI call behind applications.keyphrases_table (east_table_host =
             build + score; EAST_BENCH_E2E=two_calls: east_build_host then east_score_table_host):
             pinned host text -> device, table -> host, inside the timed region
  roofline   dominant kernel of the step: algorithmic bytes / its event-timed duration vs measured HBM peak
  cpu_baseline  the reference's own Python code (or the C port when oracle/_ref is absent) on a bounded sample

`--impl reference` times only the CPU implementation (rank 0) and prints the same line shape.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "ast-text-analysis_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "keyphrase_x_doc_scores_per_sec"
UNIT = "scores/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--docs", type=int, default=1000, help="documents per GPU")
    ap.add_argument("--doc-bytes", type=int, default=50000)
    ap.add_argument("--keyphrases", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--docs-total", type=int, default=100000, help="config4: documents of the whole job (sharded over the GPUs)")
    ap.add_argument("--gather", default="nccl", choices=["nccl", "fused"],
                    help="config4: nccl = all_gather_into_tensor (north_star); fused = the rows are stored into the other ranks' "
                         "tables by the scorer's own kernels (east_table_dev_gather, symmetric memory), one barrier ends the step")
    ap.add_argument("--gather-tiles", type=int, default=1,
                    help="config4: 1 = ONE all-gather after scoring (north_star); T > 1 = the table is scored in T document "
                         "tiles and the all-gather of tile t overlaps the scoring of tile t+1")
    ap.add_argument("--no-extras", action="store_true", help="N = 1: skip the short runs of BASELINE configs[2] and [4] "
                    "(single 200 MB document build; co-occurrence count at 10^4 x 10^5) reported under other_configs")
    ap.add_argument("--workload", default="table", choices=["table", "single_doc", "config4", "graph"],
                    help="table = BASELINE configs[1] (headline); single_doc = configs[2]: SA+LCP+annotation build "
                         "throughput of ONE document of --doc-bytes (use 200000000), replicas only for N>1")
    ap.add_argument("--cpu-sample-docs", type=int, default=0, help="0 = 2 documents per host core (max 64)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the score table of the last "
                    "device-timed step to DIR/scores.npy (float64; a seeded sample of its rows, listed in "
                    "DIR/scores_rows.npy, when the table exceeds 64 MB), so that two builds can be compared output "
                    "for output on identical inputs.  Headline workload only (--workload table, --impl b200): the "
                    "reference arm's subprocess returns timings and a checksum, not the table")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "table"):
        ap.error("--dump-outputs writes the table of --workload table with --impl b200")
    return args


def apply_env_options(_capi):
    """Tuning experiments: EAST_BENCH_OPTS="name=value,..." sets library options (east_set_option)."""
    for kv in os.environ.get("EAST_BENCH_OPTS", "").split(","):
        if "=" in kv:
            name, value = kv.split("=")
            _capi.set_option(name, int(value))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------
def cpu_sample(n_docs, doc_bytes, n_kps, procs):
    """Run oracle/run_reference.py in a subprocess (the reference's `east` package must not share an
    interpreter with the product's `east` package)."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_reference.py"), "--docs", str(n_docs),
           "--doc-bytes", str(doc_bytes), "--kps", str(n_kps), "--procs", str(procs)]
    out = subprocess.check_output(cmd, stderr=subprocess.DEVNULL, timeout=1500)
    return json.loads(out.decode().strip().splitlines()[-1])


def oracle_check(sample, kp_codes, kp_off, normalized):
    """Rows of a score table against the CPU oracle, in a subprocess (oracle/check_rows.py): the benchmark process
    itself loads nothing from oracle/.  sample: [(packed uint32 document, m, float64 row)]."""
    import tempfile
    import numpy as np
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "rows.npz")
        arrays = {"kp_codes": kp_codes, "kp_off": kp_off, "normalized": np.array(bool(normalized)), "n_rows": np.array(len(sample))}
        for i, (text, m, row) in enumerate(sample):
            arrays["text_%d" % i] = np.ascontiguousarray(text, dtype=np.uint32)
            arrays["m_%d" % i] = np.array(int(m))
            arrays["row_%d" % i] = np.ascontiguousarray(row, dtype=np.float64)
        np.savez(path, **arrays)
        out = subprocess.check_output([sys.executable, os.path.join(ROOT, "oracle", "check_rows.py"), path],
                                      stderr=subprocess.DEVNULL, timeout=1500)
    return json.loads(out.decode().strip().splitlines()[-1])


DUMP_BYTES = 64 * 10**6 - 4096   # everything --dump-outputs writes, .npy headers included, stays within 64 MB


def dump_table(out_dir, name, table):
    """out_dir/<name>.npy = table (float64 [rows, cols]).  A table larger than DUMP_BYTES is replaced by the rows of a
    fixed seeded sample, in increasing order, whose row numbers go to out_dir/<name>_rows.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    table = np.ascontiguousarray(table, dtype=np.float64)
    if table.nbytes > DUMP_BYTES:
        keep = max(1, DUMP_BYTES // (table.shape[1] * 8 + 8))
        rows = np.sort(np.random.default_rng(0).choice(table.shape[0], size=keep, replace=False))
        np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        table = table[rows]
    np.save(os.path.join(out_dir, name + ".npy"), table)


def cpu_sample_size(args):
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    docs = args.cpu_sample_docs or 2 * procs
    return docs, procs


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    docs, procs = cpu_sample_size(args)
    times, last = [], None
    for i in range(args.warmup + args.steps):
        r = cpu_sample(docs, args.doc_bytes, args.keyphrases, procs)
        if i >= args.warmup:
            times.append(r["wall_s"])
        last = r
    mean_s = sum(times) / len(times)
    value = docs * args.keyphrases / mean_s
    sample = "%d docs x %d B x %d keyphrases per step, %d processes (one task per document)" % (
        docs, args.doc_bytes, args.keyphrases, procs)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": last["kind"], "sample": sample,
                         "build_MB_per_s_per_core": last["build_MB_per_s"] / max(procs, 1)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, n_gpus):
    return {"workload": "keyphrases_table: %d keyphrases x %d synthetic Zipf docs x ~%d KB per GPU (BASELINE configs[1]), "
                        "build (SA+LCP+child+annotation) + score, normalized" % (args.keyphrases, args.docs, args.doc_bytes // 1000),
            "keyphrases": args.keyphrases, "docs_per_gpu": args.docs, "doc_bytes": args.doc_bytes,
            "parallelism": "documents sharded over %d GPU(s), all-gather of score slices (%s)" % (
                n_gpus, os.environ.get("EAST_GATHER_USED", "n/a")),
            "l2": "inputs larger than L2: packed text + sort buffers of a step are > 1 GB"}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """Samples SM clock, power and throttle reasons through NVML from a background thread
    (nvidia_ml_py; a polling nvidia-smi process measurably perturbs the step being timed)."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4), ("hw_power_brake", 0x80))

    def __init__(self, gpu_index, period_s=0.25):
        self.gpu = gpu_index
        self.period = period_s
        self.samples = []
        self.thread = None
        self.error = None
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical GPUs; map through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.gpu
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.gpu < len(ids) and ids[self.gpu].isdigit():
                    phys = int(ids[self.gpu])
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def sample(self):
        """One sample (also called from the main thread right before/after a timed region)."""
        if self.error or not hasattr(self, "handle"):
            return
        nv = self.nvml
        try:
            sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
            try:
                reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:  # noqa: BLE001
                reasons = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            power = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
            self.samples.append((time.perf_counter(), sm, reasons, power))
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)

    def _run(self):
        # NVML queries contend with CUDA API calls for driver locks: a fast poll slows the step
        # being measured several-fold, so the background poll is slow (4 Hz)
        while not self._stop.is_set() and not self.error:
            self._stop.wait(self.period)
            self.sample()

    def stop(self, t_from=None, t_to=None):
        """Summary of the samples taken in [t_from, t_to] (perf_counter clock)."""
        self._stop.set()
        if self.thread:
            self.thread.join(timeout=2)
        rows = [s for s in self.samples if (t_from is None or s[0] >= t_from) and (t_to is None or s[0] <= t_to)]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples: %s" % self.error], "samples": 0}
        sm = sorted(r[1] for r in rows)
        bits = 0
        for r in rows:
            bits |= r[2]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max,
                "reasons": [name for name, bit in self.REASONS if bits & bit],
                "power_w_max": max(r[3] for r in rows), "samples": len(rows), "source": "nvml"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import synth
    from east import _capi, utils
    from east.asts import utils as asts_utils

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own log lines (NCCL_DEBUG=VERSION/INFO on some boxes) go to a file
        os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join("/tmp", "nccl_%h_%p.log"))
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    # ---- host preprocessing (untimed, reported): generate, upper/tokenize/group, pack
    t0 = time.perf_counter()
    docs = synth.documents(args.docs, args.doc_bytes, first_seed=1 + rank * args.docs)
    t1 = time.perf_counter()
    cols = [utils.text_to_strings_collection(d) for d in docs]
    packed = [asts_utils.pack_strings_collection(c) for c in cols]
    doc_m = np.array([len(c) for c in cols], dtype=np.int32)
    doc_off = np.zeros(args.docs + 1, dtype=np.int64)
    np.cumsum([len(p) for p in packed], out=doc_off[1:])
    n_total = int(doc_off[-1])
    host_text = torch.empty(n_total, dtype=torch.int32).pin_memory()
    host_text_np = host_text.numpy().view(np.uint32)
    host_text_np[:] = np.concatenate(packed)
    # what east.relevance ships for ASCII / Latin-1 collections: one byte per code point, 0xFF ends a string
    host_text8 = torch.empty(n_total, dtype=torch.uint8).pin_memory()
    host_text8_np = host_text8.numpy()
    host_text8_np[:] = np.concatenate([asts_utils.pack_strings_collection_u8(c) for c in cols])
    kps = [utils.prepare_text(k) for k in synth.keyphrases(args.keyphrases)]
    kp_codes, kp_off = _capi.pack_keyphrases(kps)
    t2 = time.perf_counter()
    K, D = args.keyphrases, args.docs

    stream = torch.cuda.current_stream()
    text_dev = host_text.to(dev)
    kp_dev = torch.from_numpy(kp_codes.view(np.int32).copy()).to(dev)
    out_dev = torch.empty(D * K, dtype=torch.float64, device=dev)
    # N > 1: the gathered [N*D, K] table.  Default: symmetric memory, every rank's kernel stores its rows straight into
    # the tables of its peers (east_table_dev_gather: the all-gather is fused into the scoring kernel, NVLink peer
    # stores) and one symmetric-memory barrier ends the step.  EAST_BENCH_GATHER=nccl (or no symmetric memory): one
    # NCCL all_gather_into_tensor per step.
    gathered, symm = None, None
    if world > 1:
        from east import distributed as east_dist
        ok = 0
        if os.environ.get("EAST_BENCH_GATHER", "fused") == "fused" and east_dist.symmetric_memory_available():
            try:
                symm = east_dist.SymmetricTable(world * D, K, local_rank)
                ok = 1
            except Exception as e:  # noqa: BLE001
                sys.stderr.write("[rank %d] symmetric memory unavailable (%r): NCCL all-gather\n" % (rank, e))
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if not bool(flag.item()):
            symm = None
        gathered = symm.tensor.view(-1) if symm is not None else torch.empty(world * D * K, dtype=torch.float64, device=dev)
    host_out = torch.empty(D * K, dtype=torch.float64).pin_memory()
    host_out_np = host_out.numpy().reshape(D, K)
    torch.cuda.synchronize()
    os.environ["EAST_GATHER_USED"] = ("none: one GPU" if world == 1 else
                                      "fused into the scoring kernel: NVLink peer stores into symmetric memory + one barrier"
                                      if symm is not None else "one NCCL all_gather_into_tensor per step")

    debug = bool(os.environ.get("EAST_BENCH_DEBUG"))
    apply_env_options(_capi)

    # A/B: EAST_BENCH_E2E=two_calls times east_build_* followed by east_score_table_* instead of the one-call entries
    two_calls = os.environ.get("EAST_BENCH_E2E", "") == "two_calls"

    def step_device():
        ta = time.perf_counter()
        if two_calls:
            idx = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, device=local_rank,
                                              stream=stream.cuda_stream)
            tb = time.perf_counter()
            idx.score_table_dev(kp_dev.data_ptr(), kp_off, out_dev.data_ptr(), True, stream=stream.cuda_stream)
        elif symm is not None:   # east_table_dev_gather: build + score + the all-gather in one kernel
            idx = _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), kp_codes,
                                                        kp_off, symm.own_rows(rank * D), True, device=local_rank,
                                                        stream=stream.cuda_stream, peer_rows=symm.peer_rows(rank * D))
            tb = time.perf_counter()
        else:   # east_table_dev: build + score, the per-document kernel scores its document itself
            idx = _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), kp_codes,
                                                        kp_off, out_dev.data_ptr(), True, device=local_rank,
                                                        stream=stream.cuda_stream)
            tb = time.perf_counter()
        tc = time.perf_counter()
        if symm is not None and not two_calls:
            symm.barrier()             # every rank's rows have reached every table
            torch.cuda.synchronize()
        elif world > 1:
            # the step ends when the gathered [N*D, K] table is complete on this rank (without this
            # host sync the NCCL kernel of step i overlaps the build of step i+1 and both crawl)
            dist.all_gather_into_tensor(gathered, out_dev)
            torch.cuda.synchronize()
        td = time.perf_counter()
        idx.close()  # waits for the LCP / child / annotation kernels that overlapped the scorer
        info = None
        timings = idx.build_timings + getattr(idx, "score_timings", [])
        if debug:
            sys.stderr.write("[rank %d] dev step: build %.2f ms, score %.2f ms, gather %.2f ms, close %.2f ms\n" % (
                rank, (tb - ta) * 1e3, (tc - tb) * 1e3, (td - tc) * 1e3, (time.perf_counter() - td) * 1e3))
        return timings, info

    e2e_text = [host_text_np if (two_calls or os.environ.get("EAST_BENCH_E2E_WIDTH", "1") == "4") else host_text8_np]

    def step_e2e():
        ta = time.perf_counter()
        host_text_np = e2e_text[0]
        if two_calls:
            idx = _capi.DeviceIndex.build_host(host_text_np, doc_off, doc_m, device=local_rank)
            tb = time.perf_counter()
            idx.score_table_into(kp_codes, kp_off, host_out_np, True)
        elif symm is not None:   # east_table_host_gather: the same call, rows also into every rank's gathered table
            idx = _capi.DeviceIndex.build_host_and_score(host_text_np, doc_off, doc_m, kp_codes, kp_off, host_out_np,
                                                         True, device=local_rank, own_rows=symm.own_rows(rank * D),
                                                         peer_rows=symm.peer_rows(rank * D))
            tb = time.perf_counter()
        else:   # east_table_host: the call behind applications.keyphrases_table (build + score, overlapped)
            idx = _capi.DeviceIndex.build_host_and_score(host_text_np, doc_off, doc_m, kp_codes, kp_off, host_out_np,
                                                         True, device=local_rank)
            tb = time.perf_counter()
        tc = time.perf_counter()
        pipelined = idx.stat("pipelined")
        if debug:
            sys.stderr.write("e2e index: pipelined=%d miss=%d doc_sorted=%d overflow=%d\n" % (
                pipelined, idx.stat("pipeline_miss"), idx.stat("doc_sorted"), idx.stat("doc_sort_overflow")))
        if symm is not None and not two_calls:
            symm.barrier()
            torch.cuda.synchronize()
        elif world > 1:
            out_dev.copy_(host_out.view(-1), non_blocking=True)   # gather the table this step produced
            dist.all_gather_into_tensor(gathered, out_dev)
            torch.cuda.synchronize()
        idx.close()
        if debug:
            sys.stderr.write("e2e: build_host %.2f ms, score_host %.2f ms, close %.2f ms %s pipelined=%d\n" % (
                (tb - ta) * 1e3, (tc - tb) * 1e3, (time.perf_counter() - tc) * 1e3,
                [(n, round(m, 3)) for n, m in idx.build_timings], pipelined))

    # ---- algorithmic bytes of the scorer for this workload: counted once by the instrumented scorer
    idx0 = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream)
    probes = idx0.score_probes_dev(kp_dev.data_ptr(), kp_off, out_dev.data_ptr(), stream=stream.cuda_stream)
    info0 = idx0.info()
    idx0.close()
    _capi.set_option("score_bytes", probes)  # the instrumented scorer counts bytes

    # ---- keyphrase preparation (hashing / ordering / de-duplication of the query suffixes, kp_prep.cu): every
    # east_table_* call does it from scratch (one call per collection: there is nothing to reuse); the score calls
    # on an existing index keep it.  Its cost = a score call with new keyphrases minus the same call repeated.
    def timed_score(idx_, codes_):
        kd = torch.from_numpy(codes_.view(np.int32).copy()).to(dev)
        torch.cuda.synchronize()
        t_a = time.perf_counter()
        idx_.score_table_dev(kd.data_ptr(), kp_off, out_dev.data_ptr(), True, stream=stream.cuda_stream)
        torch.cuda.synchronize()
        return (time.perf_counter() - t_a) * 1e3
    idx1 = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream)
    cold, warm = [], []
    for i in range(5):
        varied = kp_codes.copy()
        varied[:: max(1, varied.size // 7)] = ord("A") + i     # other keyphrases of the same shape: a miss
        cold.append(timed_score(idx1, varied))
        warm.append(timed_score(idx1, varied))
    idx1.close()
    kp_prep_ms = max(0.0, sorted(cold)[len(cold) // 2] - sorted(warm)[len(warm) // 2])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed arm (nvidia-smi needs ~100 ms to deliver its first sample: start it before the warm-up)
    sampler = ClockSampler(local_rank)
    if not os.environ.get("EAST_BENCH_NO_SAMPLER"):
        sampler.start()
    for _ in range(args.warmup):
        step_device()
    barrier()
    t_timed0 = time.perf_counter()
    sampler.sample()
    _capi.set_option("time_kernels", 0)
    _capi.set_option("time_kernels", 2)    # event pair around the dominant kernel only: the roofline is measured live, here
    _capi.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    stage_ms = {}
    for _ in range(args.steps):
        timings, info = step_device()
        for name, ms in timings:
            stage_ms[name] = stage_ms.get(name, 0.0) + ms
    e1.record(stream)
    barrier()
    sampler.sample()
    if args.dump_outputs:
        if rank == 0:   # the [N * D, K] table as a caller of the last timed step receives it
            dump_table(args.dump_outputs, "scores", (gathered if world > 1 else out_dev).view(-1, K).cpu().numpy())
        barrier()       # the next pass's kernels of the other ranks store rows into rank 0's table: not before the copy
    launches = _capi.launch_count()
    kstats = _capi.kernel_stats()
    _capi.set_option("time_kernels", 0)
    # the table of ALL kernels of a step comes from a short instrumented pass after the timed region
    _capi.set_option("time_kernels", 1)
    table_steps = 3
    for _ in range(table_steps):
        step_device()
    barrier()
    kstats_all = _capi.kernel_stats()
    _capi.set_option("time_kernels", 0)
    dev_ms = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())

    # ---- end-to-end arm (host buffers through the C ABI)
    for _ in range(max(3, args.warmup)):   # the first host-buffer calls after a series of device-resident ones run slower
        step_e2e()
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - w0) * 1e3 / args.steps
    e2e_width = int(e2e_text[0].itemsize)
    # the same call with the text as uint32 code points (what round 1 timed; Cyrillic / CJK collections), fewer steps
    e2e_other_ms = None
    if not two_calls:
        e2e_text[0] = host_text_np if e2e_width == 1 else host_text8_np
        step_e2e()
        barrier()
        w1 = time.perf_counter()
        for _ in range(max(3, args.steps // 4)):
            step_e2e()
        barrier()
        e2e_other_ms = (time.perf_counter() - w1) * 1e3 / max(3, args.steps // 4)
        e2e_text[0] = host_text8_np if e2e_width == 1 else host_text_np
        step_e2e()   # the table the parity check reads comes from the headline variant
    # ---- from RAW TEXT: east_table_texts_host does the reference's host preprocessing (upper / tokenise / filter / group /
    # pack, utils.text_to_strings_collection) on the device too: the UTF-8 bytes of the documents go in, the table comes out
    raw_ms = None
    if not two_calls:
        raw_buf, raw_off = _capi.concat_utf8(docs)
        raw_pinned = torch.empty(raw_buf.size, dtype=torch.uint8).pin_memory()
        raw_np = raw_pinned.numpy()
        raw_np[:] = raw_buf
        raw_out = np.empty((D, K), dtype=np.float64)
        for _ in range(2):
            _capi.DeviceIndex.table_from_texts((raw_np, raw_off), kp_codes, kp_off, raw_out, True, device=local_rank).close()
        barrier()
        w2 = time.perf_counter()
        raw_steps = max(3, args.steps // 2)
        for _ in range(raw_steps):
            _capi.DeviceIndex.table_from_texts((raw_np, raw_off), kp_codes, kp_off, raw_out, True, device=local_rank).close()
        barrier()
        raw_ms = (time.perf_counter() - w2) * 1e3 / raw_steps
        raw_equal = bool(np.array_equal(raw_out.view(np.uint64), host_out_np.view(np.uint64)))
    # clocks under load: samples taken between the start of the device-timed region and the end of the e2e one
    clocks = sampler.stop(t_timed0, time.perf_counter())
    # ---- the same two arms when every call scans for its alphabet (option no_alphabet_guess): by default a batch starts
    # from the alphabet of the thread's previous batch -- a guess the per-document kernel checks code point by code point
    scanned = None
    if world == 1 and not two_calls:
        try:
            n_ab = max(8, args.steps // 2)
            scanned = {}
            for label, off_ in (("guessed", 0), ("scanned", 1)):   # both measured the same way: host wall clock, no event pairs
                _capi.set_option("no_alphabet_guess", off_)
                scanned[label] = {}
                for name, fn in (("device_ms_per_step", step_device), ("e2e_ms_per_step", step_e2e)):
                    for _ in range(3):
                        fn()
                    barrier()
                    w3 = time.perf_counter()
                    for _ in range(n_ab):
                        fn()
                    barrier()
                    scanned[label][name] = (time.perf_counter() - w3) * 1e3 / n_ab
        finally:
            _capi.set_option("no_alphabet_guess", 0)
        step_e2e()   # the table the parity check reads comes from the headline variant
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    checksum = float(host_out_np.sum())

    # ---- untimed self-check: rows of the table the LAST timed end-to-end step produced (and, at N > 1, rows of the
    # gathered table that other ranks produced) against the CPU oracle, bit for bit
    parity = {"checked": False}
    if rank == 0 and not os.environ.get("EAST_BENCH_NO_PARITY"):
        try:
            rows = sorted(set([0, 1, D // 2, D - 1] + list(range(3, D, max(1, D // 14)))))[:18]
            sample = [(packed[d], int(doc_m[d]), host_out_np[d]) for d in rows]
            other = 0
            if world > 1:
                g = gathered.view(world, D, K)
                for r in sorted(set([1, world - 1])):
                    for j in (0, D - 1):
                        col = utils.text_to_strings_collection(synth.documents(1, args.doc_bytes, first_seed=1 + r * args.docs + j)[0])
                        sample.append((asts_utils.pack_strings_collection(col), len(col), g[r, j].cpu().numpy()))
                        other += 1
            res = oracle_check(sample, kp_codes, kp_off, True)
            parity = {"checked": True, "rows_vs_oracle": len(rows), "rows_of_other_ranks": other,
                      "mismatching_rows": res["mismatching_rows"],
                      "how": "bit-exact comparison of fp64 rows with oracle/east_oracle.c (oracle/check_rows.py, a subprocess) "
                             "after the timed region"}
        except Exception as e:  # noqa: BLE001
            parity = {"checked": False, "error": repr(e)}
    if world > 1:
        gathered_sum = float(gathered.sum().item())
        local = torch.tensor([float(host_out_np.sum())], dtype=torch.float64, device=dev)
        dist.all_reduce(local)
        parity["gathered_sum"] = gathered_sum
        parity["sum_of_rank_sums"] = float(local.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel
    peak, peak_kind = load_peaks()
    traffic_table = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic_table = json.load(f)
    dom_name, dom = max(kstats.items(), key=lambda kv: kv[1]["ms"])
    per_launch_ms = dom["ms"] / max(dom["launches"], 1)
    per_launch_bytes = dom["bytes"] / max(dom["launches"], 1)
    achieved = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
    kernel_table = {k: {"launches_per_step": v["launches"] / table_steps, "ms_per_step": v["ms"] / table_steps,
                        "GBps": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 and v["bytes"] > 0 else None}
                    for k, v in sorted(kstats_all.items(), key=lambda kv: -kv[1]["ms"])}
    build_ms = sum(ms for name, ms in stage_ms.items() if name != "score") / args.steps
    score_ms = stage_ms.get("score", 0.0) / args.steps
    text_mb = args.docs * args.doc_bytes / 1e6

    tinfo = traffic_table.get(dom_name, {})
    if "dram_bytes_per_algorithmic_byte" in tinfo:   # DRAM bytes per launch from the committed ncu --set full capture
        traffic = per_launch_bytes * tinfo["dram_bytes_per_algorithmic_byte"]
    else:
        traffic = tinfo.get("dram_bytes_per_launch")
    line = {
        "metric": METRIC, "value": n_gpus * D * K / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": n_gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, n_gpus),
        "e2e": {"value": n_gpus * D * K / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(n_total * e2e_width + doc_off.nbytes + doc_m.nbytes + kp_codes.nbytes + kp_off.nbytes),
                "text_bytes_per_code_point": e2e_width,
                "from_raw_text": ({"call": "east_table_texts_host", "ms_per_step": raw_ms, "value": n_gpus * D * K / (raw_ms * 1e-3),
                                   "h2d_bytes_per_step": int(raw_off[-1]), "table_equals_e2e_table": raw_equal,
                                   "what": "UTF-8 documents in, table out: preprocessing (east/utils.py:31-79) on the device as well; "
                                           "the same preprocessing on the host costs host_prep_s.tokenize_pack"} if raw_ms else None),
                "other_width": {"text_bytes_per_code_point": 5 - e2e_width, "ms_per_step": e2e_other_ms,
                                "value": (n_gpus * D * K / (e2e_other_ms * 1e-3)) if e2e_other_ms else None},
                "d2h_bytes_per_step": int(D * K * 8),
                "call": "east_build_host+east_score_table_host" if two_calls else ("east_table_host_u8" if e2e_width == 1 else "east_table_host"),
                "keyphrase_preparation": "inside every call (device, kp_prep.cu): nothing derived from the keyphrases is cached between table calls",
                "kp_prep_ms": kp_prep_ms,
                "alphabet": "guessed: a batch starts from the alphabet of the thread's previous batch; the per-document kernel checks "
                            "every code point against it and a miss redoes the batch from a scan (tests: "
                            "test_alphabet_of_the_previous_batch_is_only_a_guess); alphabet_ab = both arms with the guess on and "
                            "switched off, measured alike (host wall clock per step, no event pairs, fewer steps)",
                "alphabet_ab": scanned},
        "parity_checked": bool(parity.get("checked") and parity.get("mismatching_rows") == 0),
        "parity": parity,
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_source": tinfo.get("source"),
                     "note": tinfo.get("note"),
                     "peak_source": peak_kind,
                     "launches_per_step": dom["launches"] / args.steps, "ms_per_launch": per_launch_ms,
                     "algorithmic_bytes_per_launch": per_launch_bytes,
                     "share_of_step": dom["ms"] / args.steps / dev_ms,
                     # the roofline that actually bounds this kernel: warp instructions issued per second against the issue
                     # peak (148 SMs x 4 schedulers x SM clock); instructions per code point from the committed ncu capture
                     "issue": ({"warp_instructions_per_code_point": tinfo["warp_instructions_per_code_point"],
                                "achieved_Ginst_per_s": tinfo["warp_instructions_per_code_point"] * n_total / (per_launch_ms * 1e-3) / 1e9,
                                "peak_Ginst_per_s": 148 * 4 * (clocks.get("sm_mhz") or 1965.0) * 1e6 / 1e9,
                                "frac": tinfo["warp_instructions_per_code_point"] * n_total / (per_launch_ms * 1e-3) /
                                        (148 * 4 * (clocks.get("sm_mhz") or 1965.0) * 1e6),
                                "active_threads_per_instruction": tinfo.get("thread_instructions_per_warp_instruction"),
                                "source": tinfo.get("instruction_source")}
                               if "warp_instructions_per_code_point" in tinfo and dom["launches"] == args.steps else None)},
        "breakdown": {"device_call": "east_build_dev+east_score_table_dev" if two_calls else "east_table_dev",
                      "build_ms": build_ms, "score_ms": score_ms,
                      "sa_build_MB_per_s": text_mb / (build_ms * 1e-3) if build_ms > 0 else None,
                      "build_codepoints_per_s": n_total / (build_ms * 1e-3) if build_ms > 0 else None,
                      "score_only_scores_per_s": D * K / (score_ms * 1e-3) if score_ms > 0 else None,
                      "stages_ms": {k: v / args.steps for k, v in stage_ms.items()},
                      "kernels": kernel_table, "scorer_algorithmic_bytes": probes,
                      "index": info0, "n_codepoints": n_total, "checksum": checksum, "kp_prep_ms": kp_prep_ms,
                      "host_prep_s": {"generate": t1 - t0, "tokenize_pack": t2 - t1}},
        "host_prep_s": {"generate": t1 - t0, "tokenize_pack": t2 - t1},
    }
    if not args.no_cpu_baseline and n_gpus == 1:
        try:
            docs_s, procs = cpu_sample_size(args)
            r = cpu_sample(docs_s, args.doc_bytes, args.keyphrases, procs)
            r1 = cpu_sample(2, args.doc_bytes, args.keyphrases, 1)
            line["cpu_baseline"] = {
                "value": r["scores_per_s"], "unit": UNIT, "cores": procs, "kind": r["kind"],
                "sample": "%d docs x %d B x %d keyphrases, %d processes, one task per document (build + score); "
                          "single process on 2 docs: %.1f scores/s" % (docs_s, args.doc_bytes, args.keyphrases, procs,
                                                                         r1["scores_per_s"]),
                "single_process_value": r1["scores_per_s"], "wall_s": r["wall_s"],
                "build_MB_per_s_per_core": r["build_MB_per_s"] / max(procs, 1)}
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(e)}
    if n_gpus == 1 and not args.no_extras:
        del text_dev, out_dev
        line["other_configs"] = extras_single_gpu(args, _capi, torch, np, synth, local_rank)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_single_doc(args):
    """BASELINE configs[2]: generalized SA + LCP + child table + annotation of one large document."""
    import numpy as np
    import torch
    import synth
    from east import _capi
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(local_rank)
    apply_env_options(_capi)
    packed, m, text_bytes, _ = synth.packed_big_document(args.doc_bytes, seed=3 + rank)
    n = int(packed.size)
    doc_off = np.array([0, n], dtype=np.int64)
    doc_m = np.array([m], dtype=np.int32)
    dev = torch.from_numpy(packed.view(np.int32)).cuda()
    stream = torch.cuda.current_stream()
    for _ in range(args.warmup):
        _capi.DeviceIndex.build_dev(dev.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream).close()
    torch.cuda.synchronize()
    _capi.set_option("time_kernels", 0)
    _capi.set_option("time_kernels", 1)
    _capi.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    stage_ms = {}
    for _ in range(args.steps):
        idx = _capi.DeviceIndex.build_dev(dev.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream)
        info = idx.info()
        idx.close()
        for name, ms in idx.build_timings:
            stage_ms[name] = stage_ms.get(name, 0.0) + ms
    e1.record(stream)
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / args.steps
    kstats = _capi.kernel_stats()
    launches = _capi.launch_count()
    _capi.set_option("time_kernels", 0)
    peak, peak_kind = load_peaks()
    dom_name, dom = max(kstats.items(), key=lambda kv: kv[1]["ms"])
    ach = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9
    print(json.dumps({
        "metric": "suffix_array_build_MB_per_sec", "value": text_bytes / 1e6 / (ms_step * 1e-3), "unit": "MB/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "replicas only", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "single document of %d text bytes: SA + LCP + child table + annotation (BASELINE configs[2])" % text_bytes,
                   "n_codepoints": n, "strings": m},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": None, "peak_source": peak_kind, "launches_per_step": dom["launches"] / args.steps},
        "breakdown": {"stages_ms": {k: v / args.steps for k, v in stage_ms.items()}, "index": info,
                      "codepoints_per_s": n / (ms_step * 1e-3),
                      "kernels": {k: {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] / args.steps}
                                  for k, v in sorted(kstats.items(), key=lambda kv: -kv[1]["ms"])}}}))


def run_config4(args):
    """BASELINE configs[3]: 10^5 keyphrases x 10^5 documents (~10 KB each; BASELINE.json gives no size), documents
    sharded over the GPUs (strong scaling: the job is fixed), per-rank [D_r, K] fp64 slices joined by ONE NCCL
    all-gather.  A step = build the rank's documents + score + all-gather; device-timed, max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import synth
    from east import _capi, utils
    from east.asts import utils as asts_utils
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join("/tmp", "nccl_%h_%p.log"))
        dist.init_process_group("nccl", device_id=dev)
    apply_env_options(_capi)
    K = args.keyphrases if args.keyphrases != 1000 else 100000
    doc_bytes = args.doc_bytes if args.doc_bytes != 50000 else 10000
    D = args.docs_total // world   # documents of this rank
    tiles = max(1, min(args.gather_tiles, D)) if world > 1 else 1
    T = (D + tiles - 1) // tiles   # documents per tile
    t0 = time.perf_counter()
    # Document ids: with one all-gather rank r owns the contiguous range [r D, (r+1) D); with tiles the table is
    # tile-major -- tile t holds documents t W T + r T + j -- so that every tile's all-gather output is one contiguous
    # block AND the gathered table is in global document order.
    texts, offs, doc_ms = [], [], []
    for t in range(tiles):
        cnt = min(T, D - t * T)
        first = (rank * D if tiles == 1 else t * world * T + rank * T)
        # numpy-only generator: the packed form of Zipf word documents without 10^5 rounds of Python tokenising
        t_t, o_t, m_t = synth.packed_collection_fast(cnt, doc_bytes, first_seed=1000003 * (t + 1) + first)
        texts.append(t_t); offs.append(np.diff(o_t)); doc_ms.append(m_t)
    doc_m = np.concatenate(doc_ms).astype(np.int32)
    doc_off = np.zeros(D + 1, dtype=np.int64)
    np.cumsum(np.concatenate(offs), out=doc_off[1:])
    host_text = np.concatenate(texts)
    text_dev = torch.from_numpy(host_text.view(np.int32)).to(dev)
    kps = [utils.prepare_text(k) for k in synth.keyphrases(K)]
    kp_codes, kp_off = _capi.pack_keyphrases(kps)
    kp_dev = torch.from_numpy(kp_codes.view(np.int32).copy()).to(dev)
    prep_s = time.perf_counter() - t0
    fused = args.gather == "fused" and world > 1 and tiles == 1
    symm = None
    if fused:
        from east import distributed as east_dist
        symm = east_dist.SymmetricTable(world * D, K, local_rank)
    out_dev = torch.empty(D * K, dtype=torch.float64, device=dev) if (tiles == 1 and not fused) else None
    bufs = [torch.empty(T * K, dtype=torch.float64, device=dev) for _ in range(2)] if tiles > 1 else None
    gathered = (symm.tensor.view(-1) if fused else torch.empty(world * D * K, dtype=torch.float64, device=dev)) if world > 1 else None
    stream = torch.cuda.current_stream()

    def step_fused():
        # ONE engine call: index, score, and the all-gather inside the scorer's kernels (peer stores over NVLink)
        idx = _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), kp_codes, kp_off,
                                                    symm.own_rows(rank * D), True, device=local_rank, stream=stream.cuda_stream,
                                                    peer_rows=symm.peer_rows(rank * D))
        symm.barrier()
        torch.cuda.synchronize()
        idx.close()
        return dict(idx.build_timings), 0.0

    def step():
        if fused:
            return step_fused()
        # every step prepares the keyphrases from scratch (suffix hashing / ordering / de-duplication on the device,
        # kp_prep.cu): a real table call is made once per collection, there is nothing to reuse
        _capi.set_option("drop_kp_cache", 1)
        idx = _capi.DeviceIndex.build_dev(text_dev.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream)
        score_ms = 0.0
        if tiles == 1:
            idx.score_table_dev(kp_dev.data_ptr(), kp_off, out_dev.data_ptr(), True, stream=stream.cuda_stream)
            score_ms = dict(idx.score_timings).get("score", 0.0)
            if world > 1:
                dist.all_gather_into_tensor(gathered, out_dev)
                torch.cuda.synchronize()
        else:
            works, base = [], 0
            for t in range(tiles):
                cnt = min(T, D - t * T)
                buf = bufs[t & 1]
                if t >= 2:
                    works[t - 2].wait()     # the collective that read this buffer two tiles ago
                idx.score_range_dev(kp_dev.data_ptr(), kp_off, t * T, cnt, buf.data_ptr(), True, stream=stream.cuda_stream)
                score_ms += dict(idx.score_timings).get("score", 0.0)
                works.append(dist.all_gather_into_tensor(gathered[base: base + world * cnt * K], buf[: cnt * K], async_op=True))
                base += world * cnt * K
            for w in works:
                w.wait()
            torch.cuda.synchronize()
        build_t = dict(idx.build_timings)
        idx.close()
        return dict(idx.build_timings) or build_t, score_ms

    for _ in range(args.warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        build_t, score_ms = step()
    e1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms_step], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item())
    checksum = float((gathered if world > 1 else out_dev)[:: max(1, D * K // 4096)].sum().item())
    full_sum = float((gathered if world > 1 else out_dev).sum().item())
    # untimed parity sample: rows of rank 0's own documents (the first rows of the table in both layouts) vs the oracle
    parity = {"checked": False}
    if rank == 0 and not os.environ.get("EAST_BENCH_NO_PARITY"):
        try:
            table = (gathered if world > 1 else out_dev)
            first_tile = min(T, D)
            rows = [0, 1, first_tile // 2, first_tile - 1]
            sample = [(host_text[doc_off[d]:doc_off[d + 1]], int(doc_m[d]), table[d * K:(d + 1) * K].cpu().numpy()) for d in rows]
            res = oracle_check(sample, kp_codes, kp_off, True)
            parity = {"checked": True, "rows_vs_oracle": len(rows), "scores_vs_oracle": len(rows) * K,
                      "mismatching_rows": res["mismatching_rows"]}
        except Exception as e:  # noqa: BLE001
            parity = {"checked": False, "error": repr(e)}
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": world * D * K / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "keyphrases_table (BASELINE configs[3]): %d keyphrases x %d synthetic Zipf docs x ~%d KB, "
                                   "documents sharded over %d GPU(s), one NCCL all-gather of the [D_r, K] fp64 slices" % (
                                       K, world * D, doc_bytes // 1000, world),
                       "keyphrases": K, "docs_total": world * D, "docs_per_gpu": D, "doc_bytes": doc_bytes,
                       "table_bytes": world * D * K * 8,
                       "gather": "fused: rows stored into the peers' tables by the scorer's kernels, one barrier" if fused else
                                 "one all-gather after scoring" if tiles == 1 else
                                 "%d document tiles, all-gather of tile t overlaps the scoring of tile t+1" % tiles},
            "parity_checked": bool(parity.get("checked") and parity.get("mismatching_rows") == 0), "parity": parity,
            "breakdown": {"build_stages_ms": build_t, "score_ms": score_ms, "host_prep_s": prep_s, "checksum_sample": checksum,
                          "table_sum": full_sum,
                          "keyphrase_preparation": "inside every timed step (device): the cache of the score calls is dropped first"}}))
    if world > 1:
        dist.destroy_process_group()


def time_cooc(_capi, torch, K, D, threshold=0.5, reps=3, device=0):
    """Kernel-only time of the co-occurrence count C = B B^T (tcgen05, cooc_tc.cu) on a random [D, K] score table."""
    g = torch.Generator(device="cuda").manual_seed(1)
    S = torch.rand((D, K), dtype=torch.float64, device="cuda", generator=g)
    C = torch.empty((K, K), dtype=torch.int32, device="cuda")
    for _ in range(2):
        _capi.cooc_dev(S.data_ptr(), D, K, threshold, C.data_ptr(), device=device)
    _capi.set_option("time_kernels", 0); _capi.set_option("time_kernels", 1)
    for _ in range(reps):
        _capi.cooc_dev(S.data_ptr(), D, K, threshold, C.data_ptr(), device=device)
    ks = _capi.kernel_stats(); _capi.set_option("time_kernels", 0)
    per = {k: v["ms"] / max(v["launches"], 1) for k, v in ks.items()}
    gemm = per.get("k_cooc_umma_tma") or per.get("k_cooc_umma_pipe") or per.get("k_cooc_umma")
    # spot check against a dense fp32 product of a slab (exact in fp32: counts < 2^24)
    Bs = (S[:, :256] >= threshold).to(torch.float32)
    ref = (Bs.t() @ Bs).to(torch.int32)
    ok = bool(torch.equal(ref, C[:256, :256]))
    del S, C
    return {"K": K, "D": D, "kernels_ms": per, "gemm_ms": gemm, "ops": 2.0 * K * K * D,
            "TOPS_on_full_product": 2.0 * K * K * D / (gemm * 1e-3) / 1e12 if gemm else None,
            "TOPS_executed": 2.0 * K * K * D * 0.5 * (1 + 256.0 / K) / (gemm * 1e-3) / 1e12 if gemm else None,
            "slab_exact_vs_fp32_matmul": ok}


def extras_single_gpu(args, _capi, torch, np, synth, local_rank):
    """Short untimed-region extras for the N = 1 line: BASELINE configs[2] (one 200 MB document: SA + LCP + child table
    + annotation build throughput) and the tensor-core half of configs[4] (co-occurrence count at 10^4 x 10^5)."""
    out = {}
    try:
        packed, m, text_bytes, _ = synth.packed_big_document(200_000_000, seed=3)
        n = int(packed.size)
        doc_off = np.array([0, n], dtype=np.int64)
        doc_m = np.array([m], dtype=np.int32)
        dev_text = torch.from_numpy(packed.view(np.int32)).cuda()
        stream = torch.cuda.current_stream()
        for _ in range(2):
            _capi.DeviceIndex.build_dev(dev_text.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream).close()
        torch.cuda.synchronize()
        _capi.set_option("time_kernels", 0); _capi.set_option("time_kernels", 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        reps = 3
        for _ in range(reps):
            _capi.DeviceIndex.build_dev(dev_text.data_ptr(), doc_off, doc_m, device=local_rank, stream=stream.cuda_stream).close()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        ks = _capi.kernel_stats(); _capi.set_option("time_kernels", 0)
        peak, _ = load_peaks()
        sweep = ks.get("k_rs_onesweep")
        out["single_doc_200MB"] = {
            "metric": "suffix_array_build_MB_per_sec", "value": text_bytes / 1e6 / (ms * 1e-3), "unit": "MB/s", "ms_per_build": ms,
            "text_bytes": text_bytes, "n_codepoints": n, "strings": m, "codepoints_per_s": n / (ms * 1e-3),
            "what": "BASELINE configs[2]: SA + LCP + child table + annotation of ONE document (global prefix-doubling sort), device-timed",
            "k_rs_onesweep": ({"launches_per_build": sweep["launches"] / reps, "ms_per_build": sweep["ms"] / reps,
                               "GBps": sweep["bytes"] / (sweep["ms"] * 1e-3) / 1e9,
                               "frac_of_hbm_peak": sweep["bytes"] / (sweep["ms"] * 1e-3) / 1e9 / peak} if sweep else None),
            "kernels_ms": {k: v["ms"] / reps for k, v in sorted(ks.items(), key=lambda kv: -kv[1]["ms"])[:8]}}
        del dev_text
    except Exception as e:  # noqa: BLE001
        out["single_doc_200MB"] = {"error": repr(e)}
    try:
        _capi.trim(local_rank)
        out["cooccurrence_1e4x1e5"] = time_cooc(_capi, torch, 10000, 100000, device=local_rank)
        out["cooccurrence_1e4x1e5"]["what"] = ("BASELINE configs[4], tensor-core half: C = B B^T of 10^4 keyphrases x 10^5 documents "
                                               "(tcgen05.mma kind::i8), kernel time from CUDA events")
    except Exception as e:  # noqa: BLE001
        out["cooccurrence_1e4x1e5"] = {"error": repr(e)}
    _capi.trim(local_rank)
    return out


def run_graph(args):
    """BASELINE configs[4]: keyphrases graph (-r 0.25 -c 0.6) over 10^4 keyphrases x 10^5 documents (~10 KB), documents
    sharded over the GPUs.  A step = index + score this rank's documents (east_table_dev), count the co-occurrences of
    its rows on the tensor cores (C_r = B_r B_r^T, east_cooc_dev), ONE all-reduce (int32 sum) of the K x K counts.
    Device-timed, max over ranks.  The graph dict itself (K^2 confidences) is assembled on the host from C, untimed."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import synth
    from east import _capi, utils
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join("/tmp", "nccl_%h_%p.log"))
        dist.init_process_group("nccl", device_id=dev)
    apply_env_options(_capi)
    K = args.keyphrases if args.keyphrases != 1000 else 10000
    doc_bytes = args.doc_bytes if args.doc_bytes != 50000 else 10000
    D = args.docs_total // world
    t0 = time.perf_counter()
    host_text, doc_off, doc_m = synth.packed_collection_fast(D, doc_bytes, first_seed=77 + rank * 1009)
    text_dev = torch.from_numpy(host_text.view(np.int32)).to(dev)
    names = synth.keyphrases(K)
    kp_codes, kp_off = _capi.pack_keyphrases([utils.prepare_text(k) for k in names])
    kp_dev = torch.from_numpy(kp_codes.view(np.int32).copy()).to(dev)
    prep_s = time.perf_counter() - t0
    S = torch.empty(D * K, dtype=torch.float64, device=dev)
    C = torch.empty((K, K), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    r_thr, c_conf = 0.25, 0.6

    def step():
        ev[0].record(stream)
        _capi.DeviceIndex.build_dev_and_score(text_dev.data_ptr(), doc_off, doc_m, kp_dev.data_ptr(), kp_codes, kp_off,
                                              S.data_ptr(), True, device=local_rank, stream=stream.cuda_stream).close()
        ev[1].record(stream)
        _capi.cooc_dev(S.data_ptr(), D, K, r_thr, C.data_ptr(), device=local_rank, stream=stream.cuda_stream)
        ev[2].record(stream)
        if world > 1:
            dist.all_reduce(C, op=dist.ReduceOp.SUM)
        ev[3].record(stream)
        torch.cuda.synchronize()
        return [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]

    for _ in range(args.warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    parts = np.zeros(3)
    for _ in range(args.steps):
        parts += np.array(step())
    e1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms_step], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item())
    parts /= args.steps
    # untimed: the graph itself + checks (support = diagonal; symmetric; a slab against a dense fp32 product of rank 0's rows
    # is only exact at N = 1, so the check there is on the all-reduced diagonal instead)
    support = torch.diagonal(C).to(torch.int64)
    local_support = (S.view(D, K) >= r_thr).sum(dim=0).to(torch.int64)
    if world > 1:
        dist.all_reduce(local_support, op=dist.ReduceOp.SUM)
    checks = {"support_equals_column_counts": bool(torch.equal(support, local_support)),
              "symmetric": bool(torch.equal(C[:512, :512], C[:512, :512].t()))}
    if rank == 0:
        from east import applications
        t1 = time.perf_counter()
        graph = applications.graph_from_cooccurrence(names, names, C.cpu().numpy(), c_conf, r_thr, 1)
        graph_s = time.perf_counter() - t1
        print(json.dumps({
            "metric": METRIC, "value": world * D * K / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64 scores, u8 x u8 -> s32 co-occurrence", "data": "synthetic",
            "config": {"workload": "keyphrases_graph -r %.2f -c %.2f (BASELINE configs[4]): %d keyphrases x %d synthetic Zipf docs x ~%d KB, "
                                   "documents sharded over %d GPU(s); per rank build + score + tensor-core co-occurrence, one all-reduce "
                                   "of the K x K int32 counts" % (r_thr, c_conf, K, world * D, doc_bytes // 1000, world),
                       "keyphrases": K, "docs_total": world * D, "docs_per_gpu": D, "doc_bytes": doc_bytes},
            "parity_checked": all(checks.values()), "parity": checks,
            "breakdown": {"table_ms": parts[0], "cooc_ms": parts[1], "all_reduce_ms": parts[2],
                          "cooc_TOPS_on_full_product": 2.0 * K * K * D / (parts[1] * 1e-3) / 1e12,
                          "graph_nodes": len(graph["nodes"]), "graph_edges": len(graph["edges"]), "graph_assembly_host_s": graph_s,
                          "host_prep_s": prep_s}}))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: whatever a library prints there on its own (NCCL's version line under
    # NCCL_DEBUG=VERSION, for one) is sent to stderr -- the process's descriptor 1 points at stderr while the run lasts,
    # and print() below writes to a copy of the real one
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w", buffering=1)   # line-buffered: the JSON line leaves with its newline
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.workload == "config4" and args.impl == "b200":
        return run_config4(args)
    if args.workload == "single_doc" and args.impl == "b200":
        return run_single_doc(args)
    if args.workload == "graph" and args.impl == "b200":
        return run_graph(args)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
