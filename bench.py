#!/usr/bin/env python3
"""bench.py -- genotypes scored per second on B200, the metric of BASELINE.json.

Workload (config.workload): BASELINE.json configs[2], the synthetic genome-wide PRS of
1,000,000 variants x 500,000 samples, variant-sharded.  It does not fit one GPU (1 TB of int8
GT), so every rank holds the per-GPU shard of the 8-GPU run -- 125,000 variants x 500,000
samples = 125 GB of raw BCF GT bytes resident in HBM -- and N ranks score N such shards (weak
scaling; N = 8 is the whole problem).  One step = one pass of the scoring path over the rank's
shard (count -> decide -> accumulate for every score row) followed by the cross-rank combine
of the per-sample partial sums.

value    : genotypes/s, whole job, inputs resident in HBM when the timed region starts.
e2e      : same metric through npc_score_block with HOST buffers: pinned staging -> H2D ->
           kernels -> D2H of the scores, every step, on a bounded slice of the same cohort.
roofline : algorithmic HBM bytes (2 B per genotype + row metadata + sums traffic) / measured time
           of the scoring kernels, against MEASURED_PEAKS.json hbm_gbs.
cpu_baseline : the CPU oracle (a C port of the reference algorithm; the Nim reference cannot be
           built in this image) on a bounded sample of the same cohort.
--impl reference : that oracle with all host threads, as the reference arm.
--dump-outputs DIR : after the timed steps, what the headline's last step computed, as DIR/<name>.npy (see dump_outputs);
           the inputs are a pure function of the arguments, so two builds can be compared output for output.
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
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

SEED = 0x6E696D70
N_SAMPLES = 500_000
V_PER_GPU = 125_000
MISS_RATE = 0.005
DUMP_BYTES = 60_000_000                 # --dump-outputs: data bytes in all, under 64 MB with the .npy headers


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples", type=int, default=N_SAMPLES)
    ap.add_argument("--variants", type=int, default=V_PER_GPU, help="variants per GPU (shard)")
    ap.add_argument("--block-rows", type=int, default=0, help="score rows per npc_score_block_device call (0 = auto)")
    ap.add_argument("--e2e-variants", type=int, default=4096)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--brief", action="store_true", help="print value / roofline / shape only (tuning sweeps)")
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5],
                    help="BASELINE.json config to time as the headline (default 3: the genome-wide shard)")
    ap.add_argument("--no-extra", action="store_true", help="skip the short timings of configs 2, 4 and 5 (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm sizes its sample from a calibration timing, so its outputs differ from run to run")
    return args


def locus_fields(loci):
    """The per-locus records (nb.LOCUS_DTYPE, any shape) as one array per field."""
    return {"loci_" + f: loci[f] for f in ("klass", "used", "eaidx", "ngt", "nmiss", "neff", "imputed")}


def dump_outputs(path, arrays):
    """Write every array as <path>/<name>.npy in float64 (the integer fields are exact there).  When they hold more
    than DUMP_BYTES in all, each array larger than an equal share keeps a sample of that many positions, drawn from a
    generator seeded by SEED and the array's size and kept in order: the same positions in every run."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    share = DUMP_BYTES // 8 // len(arrays)
    sample = sum(a.size for a in arrays.values()) * 8 > DUMP_BYTES
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if sample and a.size > share:
            a = a.ravel()[np.sort(np.random.default_rng([SEED, a.size]).choice(a.size, share, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


# ---- synthetic score rows / cohort parameters (SURVEY.md 8d) -------------------------------------

def cohort_params(v0, V):
    """Per-variant parameters as a pure function of the variant index: af ~ U(0.01, 0.5),
    beta ~ N(0, 0.05^2) rounded to 4 decimals, eaf = af rounded, ref == ea for 27% of rows."""
    rng = np.random.default_rng([SEED, v0])
    af = rng.uniform(0.01, 0.5, size=V)
    beta = np.round(rng.normal(0.0, 0.05, size=V), 4)
    ref_is_ea = (rng.random(V) < 0.27).astype(np.int32)
    af_thr = (af * 65536).astype(np.uint32)
    miss_thr = np.full(V, int(MISS_RATE * (1 << 24)), dtype=np.uint32)
    alt = np.ones(V, dtype=np.int32)
    return af, beta, ref_is_ea, af_thr, miss_thr, alt


def make_rows(dtype, V, af, beta, ref_is_ea):
    rows = np.zeros(V, dtype=dtype)
    rows["gt_row"] = np.arange(V)
    rows["ref_is_ea"] = ref_is_ea
    rows["eaidx"] = np.where(ref_is_ea == 1, 0, 1)
    rows["beta"] = beta
    rows["eaf"] = np.round(af, 4)
    rows["kind"] = 0
    return rows


# ---- clocks -------------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi clocks + throttle reasons of one GPU, sampled every 50 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU oracle legs ------------------------------------------------------------------------------

def cpu_oracle_rate(n, seconds, threads):
    """Time the oracle (tests/orc.py -> oracle/nimpress_oracle.c) on a bounded sample of the same
    cohort: first a calibration batch, then enough variants for about `seconds` of work."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orc
    stride = -(-2 * n // 128) * 128

    def run(V):
        af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(0, V)
        gt = np.zeros((V, stride), dtype=np.int8)
        orc.synth_fill(gt, n, 0, SEED, af_thr, miss_thr, alt)
        rows = make_rows(orc.ROW_DTYPE, V, af, beta, ref_is_ea)
        t0 = time.perf_counter()
        out = orc.score_matrix(gt, n, 2, rows, threads=threads)
        dt = time.perf_counter() - t0
        assert out["nloci"] == V
        return dt, out["loci"], rows

    v_cal = max(threads * 4, 16)
    dt, _, _ = run(v_cal)
    V = int(min(max(v_cal, seconds / max(dt, 1e-6) * v_cal), 40_000, (24 << 30) // stride))
    V = max(V - V % threads, threads)
    dt, loci, rows = run(V)
    cpu_oracle_rate.last = (loci, rows)
    return n * V / dt, V, dt


def cpu_af_test_ms_per_locus(n, max_loci=24):
    """The reference also runs binomTest(neff, 2*(n - nmiss), eaf) per matched locus for its AF-mismatch
    warning (src/nimpress.nim:573; an O(n) enumeration, :155-188).  Timed here on the tallies of the
    loci just scored, single thread like the reference, so that the CPU baseline can be quoted with
    and without it (SURVEY section 8d)."""
    import orc
    loci, rows = cpu_oracle_rate.last
    L = orc.lib()
    k = min(max_loci, len(loci))
    t0 = time.perf_counter()
    for i in range(k):
        L.orc_binom_test(int(loci["neff"][i]), int(2 * (n - loci["nmiss"][i])), float(rows["eaf"][i]))
    return (time.perf_counter() - t0) * 1e3 / max(k, 1)


def reference_arm(args):
    """--impl reference: the CPU implementation of the path (the oracle port; the Nim reference
    cannot be compiled here) with all host threads, on bounded samples of this workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.samples
    rates, sample_v, ms = [], 0, []
    per_step = max(args.cpu_seconds / max(args.steps + args.warmup, 1), 2.0)
    for i in range(args.warmup + args.steps):
        r, V, dt = cpu_oracle_rate(n, per_step, threads)
        if i >= args.warmup:
            rates.append(r); sample_v = V; ms.append(dt * 1e3)
    value = float(np.mean(rates))
    line = {
        "impl": "reference", "metric": "genotypes scored/sec (variants x samples)", "value": value,
        "unit": "genotypes/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(ms)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"config3 shard: {n} samples, bounded sample of {sample_v} variants per step",
                   "samples": n, "variants_per_step": sample_v},
        "cpu_baseline": {"value": value, "unit": "genotypes/s", "cores": threads, "kind": "port",
                         "sample": f"{sample_v} variants x {n} samples per step, rows split over {threads} threads, "
                                   "AF-mismatch binomTest (warning only) not run"},
        "e2e": {"value": value, "unit": "genotypes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---- the other BASELINE configs, timed briefly (N = 1) ---------------------------------------------

def time_resident(nb, torch, dev, n, V, miss_lo, miss_hi, steps=20, warmup=5, policy=None):
    """Kernel-only rate of one npc_score_block_device call over a resident V x n slab (CUDA events around the
    call, L2 flushed by a 512 MB write before every timed call: these slabs are near or below the L2 size)."""
    stride = -(-2 * n // 128) * 128
    af, beta, ref_is_ea, af_thr, _, alt = cohort_params(0, V)
    rng = np.random.default_rng([SEED, 99])
    miss_thr = (rng.uniform(miss_lo, miss_hi, size=V) * (1 << 24)).astype(np.uint32)
    rows = make_rows(nb.ROW_DTYPE, V, af, beta, ref_is_ea)
    eng = nb.Engine(n, max_rows_per_block=V, n_slots=0, device=dev.index)
    stream = torch.cuda.current_stream(dev)
    eng.set_stream(stream.cuda_stream)
    eng.set_policy(**(policy or {}))
    gt = torch.empty((V, stride), dtype=torch.uint8, device=dev)
    eng.synth_fill_device(gt, stride, 0, V, SEED, torch.from_numpy(af_thr.view(np.int32)).to(dev),
                          torch.from_numpy(miss_thr.view(np.int32)).to(dev), torch.from_numpy(alt).to(dev))
    d_rows = torch.from_numpy(rows.view(np.uint8).reshape(V, -1)).to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    ms = []
    t_warm = time.perf_counter()                        # the GPU may have idled through the CPU legs: launches for 0.3 s bring the clocks back up
    while time.perf_counter() - t_warm < 0.3:
        eng.reset()
        eng.score_block_device(gt, stride, V, d_rows, n_rows=V)
        torch.cuda.synchronize()
    for i in range(warmup + steps):
        eng.reset()
        flush.fill_(i & 255)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.score_block_device(gt, stride, V, d_rows, n_rows=V)
        e1.record(stream)
        torch.cuda.synchronize()
        if i >= warmup:
            ms.append(e0.elapsed_time(e1))
    out = eng.finish(want_loci=True)
    shape = eng.kernel_shape_for(V)
    eng.close()
    t = float(np.median(ms)) * 1e-3
    return t, out, shape, 2.0 * n * V + 32.0 * V + 16.0 * n


def extra_configs(nb, torch, dev, peak, steps=None, warmup=None):
    """configs[1], [3] and [4] of BASELINE.json, a few launches each -> (timings, outputs of each config's last call).
    steps / warmup: timed and untimed calls of each config (None: 20 / 5 launches of configs 2 and 5, 5 / 1 calls of
    config 4, the short timings beside the genome-wide headline)."""
    ex, outs = {}, {}
    reps = {} if steps is None else dict(steps=steps, warmup=warmup)
    t, out, shape, alg = time_resident(nb, torch, dev, 100_000, 697, 0.005, 0.005, **reps)
    outs["config2"] = {"scores": out["scores"], "nloci": out["nloci"], **locus_fields(out["loci"])}
    ex["config2"] = {"workload": "697 loci (the wood height score's size) x 100,000 samples, 0.5% missing, one launch",
                     "value": 100_000 * 697 / t, "unit": "genotypes/s", "launch_us": t * 1e6, "roofline_frac": alg / t / 1e9 / peak,
                     "grid": shape["grid"], "row_groups": shape.get("row_groups"), "l2": "flushed before every timed launch"}
    t, out, shape, alg = time_resident(nb, torch, dev, 50_000, 10_000, 0.0, 0.10, **reps)
    outs["config5"] = {"scores": out["scores"], "nloci": out["nloci"], **locus_fields(out["loci"])}
    ex["config5"] = {"workload": "10,000 loci x 50,000 samples, per-locus missing rate U(0, 0.10), --maxmis 0.05 (default policies), one launch",
                     "value": 50_000 * 10_000 / t, "unit": "genotypes/s", "launch_us": t * 1e6, "roofline_frac": alg / t / 1e9 / peak,
                     "loci_over_maxmis": int((out["loci"]["klass"] == 4).sum()), "grid": shape["grid"], "row_groups": shape.get("row_groups"),
                     "l2": "flushed before every timed launch"}
    # config 4: 18 score definitions over one resident slab in one call (tensor-core contraction)
    n, V, S = 200_000, 20_000, 18
    stride = -(-2 * n // 128) * 128
    af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(0, V)
    base = make_rows(nb.ROW_DTYPE, V, af, beta, ref_is_ea)
    rng = np.random.default_rng(7)
    lists = []
    for k in range(S):
        r = base.copy()
        r["beta"] = np.round(rng.normal(0, 0.05, V), 4)
        lists.append(r)
    eng = nb.Engine(n, max_rows_per_block=V, n_slots=0, device=dev.index)
    gt = torch.empty((V, stride), dtype=torch.uint8, device=dev)
    eng.synth_fill_device(gt, stride, 0, V, SEED, torch.from_numpy(af_thr.view(np.int32)).to(dev),
                          torch.from_numpy(miss_thr.view(np.int32)).to(dev), torch.from_numpy(alt).to(dev))
    torch.cuda.synchronize()
    eng.resident_adopt(gt, stride, V)
    pin_s = torch.empty((S, n), dtype=torch.float64).pin_memory()
    pin_l = torch.empty((S, V * nb.LOCUS_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
    sc_out = [pin_s[k].numpy() for k in range(S)]
    lo_out = [pin_l[k].numpy().view(nb.LOCUS_DTYPE) for k in range(S)]
    ts = []
    steps4, warmup4 = (5, 1) if steps is None else (steps, warmup)
    for rep in range(warmup4 + steps4):
        t0 = time.perf_counter()
        nloci4 = [nl for _, nl, _ in eng.score_resident_multi(lists, [0.0] * S, sc_out, lo_out)]
        ts.append(time.perf_counter() - t0)
    t = float(np.median(ts[warmup4:]))
    outs["config4"] = {"scores": np.stack(sc_out), "nloci": nloci4, **locus_fields(np.stack(lo_out))}
    ex["config4"] = {"workload": f"{S} score definitions x {V} loci x {n} samples over one resident 8 GB slab, one npc_score_resident_multi call "
                                 "(wall clock: row tables H2D, tally + contraction kernels, 18 x n scores and records D2H)",
                     "value": float(V) * n * S / t, "unit": "genotype-score cells/s", "call_ms": t * 1e3,
                     "slab_reads_per_s_gb": 2.0 * V * n / t / 1e9, "contractions_served": int(eng.multi_contractions),
                     "substitution": "BASELINE names 18 bundled score files; 4 of the bundled files are score definitions, so 18 synthetic "
                                     "definitions over one site set stand in (DESIGN.md section 7)"}
    eng.close()
    return ex, outs


# ---- B200 arm -------------------------------------------------------------------------------------

def b200_arm(args):
    import torch
    import torch.distributed as dist
    import nimpress_b200 as nb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    if args.config in (2, 4, 5):
        # the small configs are single launches near or below the L2 size: timed one launch at a time with the L2 flushed
        # in between (time_resident / extra_configs), N = 1 only
        if world > 1:
            raise SystemExit("--config 2 / 4 / 5 are single-GPU configurations")
        stream = torch.cuda.Stream(device=dev)
        torch.cuda.set_stream(stream)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
        ex, outs = extra_configs(nb, torch, dev, peak, args.steps, args.warmup)
        ex, outs = ex[f"config{args.config}"], outs[f"config{args.config}"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outs)
        line = {"metric": "genotypes scored/sec (variants x samples)", "value": ex["value"], "unit": ex["unit"], "n_gpus": 1,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ex.get("launch_us", ex.get("call_ms", 0.0) * 1e3) / 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": ex["workload"], "l2": ex.get("l2", "8 GB slab: larger than L2")},
                "roofline": {"bound": "hbm", "frac": ex.get("roofline_frac"), "peak": peak, "unit": "GB/s"}, "detail": ex}
        print(json.dumps(line))
        return
    n, V = args.samples, args.variants
    stride = -(-2 * n // 128) * 128
    fused = os.environ.get("NPC_FUSED", "1") != "0"
    # fused kernel: one persistent launch per block, any size; two-kernel path: ~48 MB tiles so
    # that the accumulate pass finds the tile in L2
    block_rows = args.block_rows or (min(V, 32768) if fused else max(1, min(V, (48 << 20) // stride)))
    v0 = rank * V                                                             # this rank's slice of the variant axis
    af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(v0, V)
    rows = make_rows(nb.ROW_DTYPE, V, af, beta, ref_is_ea)

    eng = nb.Engine(n, max_rows_per_block=max(block_rows, 1), n_slots=0, device=local)
    shape = eng.kernel_shape_for(min(block_rows, V))
    # a real (non-default) stream: the default stream's handle is 0, which npc_set_stream reads as
    # "use the context's own stream" and the timing events below would then miss the kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)
    eng.set_policy()                                                          # nimpress defaults
    gt = torch.empty((V, stride), dtype=torch.uint8, device=dev)
    t_af = torch.from_numpy(af_thr.view(np.int32)).to(dev)
    t_ms = torch.from_numpy(miss_thr.view(np.int32)).to(dev)
    t_alt = torch.from_numpy(alt).to(dev)
    eng.synth_fill_device(gt, stride, v0, V, SEED, t_af, t_ms, t_alt)
    # block-relative row tables, resident on the device (inputs are in HBM before the clock starts)
    rows_rel = rows.copy()
    rows_rel["gt_row"] = np.arange(V) % block_rows
    d_rows = torch.from_numpy(rows_rel.view(np.uint8).reshape(V, -1)).to(dev)
    torch.cuda.synchronize()

    class _Wrap:   # expose library-owned device memory to torch without a copy
        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 3}

    def new_comm(e):
        """NCCL communicator of the C ABI (npc_comm_init): rank 0's id reaches the others over torch.distributed."""
        ident = [nb.Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        e.comm_init(ident[0], rank, world)

    if world > 1:
        new_comm(eng)
        sums_ptr, nloci_ptr = eng.combined_device_ptr()         # combined sums / nloci after npc_comm_combine
    else:
        sums_ptr, nloci_ptr = eng.partial_device_ptr()
    t_sums = torch.as_tensor(_Wrap(sums_ptr, (n,), "<f8"), device=dev)
    t_nloci = torch.as_tensor(_Wrap(nloci_ptr, (1,), "<i8"), device=dev)

    launch_events = []                                  # (start, end, rows) of every scoring launch of the timed steps

    def step(timed=False):
        eng.reset()
        for r0 in range(0, V, block_rows):
            nr = min(block_rows, V - r0)
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
            eng.score_block_device(gt[r0], stride, nr, d_rows[r0], n_rows=nr)
            if timed:
                e1.record(stream)
                launch_events.append((e0, e1, nr))
        if world > 1:                                  # npc_comm_combine: all-gather over NCCL/NVLink, add in rank order, on the stream
            eng.comm_combine(offset=None, want_scores=False)
        return t_sums, t_nloci

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record(stream)
    for i in range(args.steps):
        total, nl = step(timed=True)
        ev[i + 1].record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.launches - l0
    ms_total = ev[0].elapsed_time(ev[-1])
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    genotypes_step = float(n) * V * world
    value = genotypes_step / (ms_step * 1e-3)
    assert int(nl.item()) == V * world, (int(nl.item()), V * world)
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path holds after the last step: the per-sample sums (combined over the ranks when
        # N > 1), nloci, and the per-locus records of this rank's shard
        dump_outputs(args.dump_outputs, {"sums": total.cpu().numpy(), "nloci": nl.cpu().numpy(),
                                         **locus_fields(eng.partial(want_loci=True)["loci"])})

    # N > 1: the combine is checked, not assumed.  Every rank scores the first Vp rows of its shard into a
    # fresh context and the ranks combine them through the same npc_comm_combine; rank 0 then scores every
    # rank's Vp rows ALONE on its own GPU (the cohort is a pure function of the variant index) and adds the
    # partial sums in rank order on the host: the two must agree bit for bit, nloci included.
    parity_checked = None
    if world > 1:
        Vp = min(512, V)
        pe = nb.Engine(n, max_rows_per_block=Vp, n_slots=0, device=local)
        pe.set_policy(); pe.reset()
        new_comm(pe)
        pe.score_block_device(gt[0], stride, Vp, rows_rel[:Vp])
        comb, comb_nl = pe.comm_combine(offset=None)
        pe.close()
        if rank == 0:
            total, total_nl = None, 0
            small = torch.empty((Vp, stride), dtype=torch.uint8, device=dev)
            for k in range(world):
                afk, betak, refk, afthr_k, missthr_k, altk = cohort_params(k * V, V)
                rk = make_rows(nb.ROW_DTYPE, V, afk, betak, refk)[:Vp]
                e = nb.Engine(n, max_rows_per_block=Vp, n_slots=0, device=local)
                e.set_policy(); e.reset()
                e.synth_fill_device(small, stride, k * V, Vp, SEED, torch.from_numpy(afthr_k[:Vp].view(np.int32).copy()).to(dev),
                                    torch.from_numpy(missthr_k[:Vp].view(np.int32).copy()).to(dev), torch.from_numpy(altk[:Vp].copy()).to(dev))
                e.score_block_device(small, stride, Vp, rk)
                pk = e.partial()
                total = pk["sums"] if total is None else total + pk["sums"]
                total_nl += pk["nloci"]
                e.close()
            same = np.array_equal(comb.view(np.uint64), total.view(np.uint64)) and comb_nl == total_nl
            assert same, "N-GPU combine differs from the rank-order sum of the shards scored alone"
            parity_checked = True
            del small

    # roofline of the dominant kernel on this rank: algorithmic bytes per launch (SURVEY.md 8d:
    # 2 B per genotype + 32 B per row + 16 B per sample per launch) / mean duration of the full-size
    # launches, measured with CUDA events on the launching stream inside the timed region
    full = [(a.elapsed_time(b), r) for a, b, r in launch_events if r == min(block_rows, V)]
    launch_ms = float(np.mean([t for t, _ in full]))
    launch_rows = full[0][1]
    alg_bytes = 2.0 * n * launch_rows + 32.0 * launch_rows + 16.0 * n
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tile_ver = 4 if os.environ.get("NPC_TILE_V") == "4" else 5
    tpath = os.path.join(ROOT, "profiles", "traffic.json")          # dram bytes of one ncu --set full capture of this launch shape
    if os.path.exists(tpath):
        for t in json.load(open(tpath)):
            if (t["samples"] == n and t["rows"] == launch_rows and t["fused"] == shape["fused"] and t.get("ver", 5) == tile_ver
                    and t.get("row_groups", 1) == shape.get("row_groups", 1)):
                traffic, traffic_src = t["dram_bytes"], t["source"]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "launch_ms": launch_ms, "rows_per_launch": launch_rows, "launches_per_step": len(launch_events) // args.steps,
                "kernel": {2: ("k_fused_pair" if tile_ver == 5 else "k_fused_tile4") + " (count+decide+accumulate, one persistent launch per block)",
                           1: ("k_fused_pair" if tile_ver == 5 else "k_fused_tile4") + " in exact-order mode (one persistent launch per block)",
                           3: "k_count_i8x2 + k_decide, then k_fused_pair in decided mode per sample slab (cohort too wide for one resident pass)",
                           0: "k_count_i8x2 + k_decide + k_accum_i8x2 sequence"}[shape["fused"]],
                "algorithmic_bytes_per_launch": alg_bytes}

    # end to end through the staged C-ABI call with HOST buffers: every step the rows are copied from ordinary
    # (pageable) host memory -- where a reader leaves the decoded BCF GT payloads -- into the pinned slot the
    # library lends, by a few host threads, then H2D -> kernels, and the scores come back D2H.  The fill is
    # inside the timed region (round 1 timed pre-filled slots).
    e2e = None
    if not args.no_e2e:
        from concurrent.futures import ThreadPoolExecutor
        Ve = min(args.e2e_variants, V)
        eb = max(1, min(Ve, (256 << 20) // stride))
        e_eng = nb.Engine(n, max_rows_per_block=eb, n_slots=3, device=local)
        e_eng.set_policy()
        host_rows = rows[:Ve].copy()
        host_rows["gt_row"] = np.arange(Ve) % eb
        host_gt = gt[:Ve].cpu().numpy()                 # the host's copy of the rows (pageable memory)
        T = max(1, min(8, (os.cpu_count() or 1) // max(world, 1)))
        pool = ThreadPoolExecutor(T)
        scores_host = None

        def fill(view, r0, nr):                         # numpy releases the GIL inside the copies
            cuts = [nr * k // T for k in range(T + 1)]
            list(pool.map(lambda k: np.copyto(view[cuts[k]:cuts[k + 1], :stride], host_gt[r0 + cuts[k]:r0 + cuts[k + 1]]), range(T)))

        def e2e_step(with_fill):
            e_eng.reset()
            for r0 in range(0, Ve, eb):
                nr = min(eb, Ve - r0)
                s, view = e_eng.stage_acquire()         # blocks until the slot's previous block is done
                if with_fill:
                    fill(view, r0, nr)
                e_eng.score_block(s, nr, host_rows[r0:r0 + nr])
            return e_eng.finish(want_loci=False)["scores"]

        def timed(with_fill):
            nonlocal scores_host
            for _ in range(max(args.warmup, 1)):
                e2e_step(with_fill)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                scores_host = e2e_step(with_fill)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / args.steps
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        dt_fill = timed(True)                           # leaves every pinned slot holding real rows of the cohort
        dt = timed(False)
        e2e = {"value": float(n) * Ve * world / dt, "unit": "genotypes/s",
               "h2d_bytes_per_step": int(stride) * Ve + 32 * Ve, "d2h_bytes_per_step": 8 * n + 8,
               "variants_per_step": Ve, "ms_per_step": dt * 1e3,
               "note": "per rank and step: npc_stage_acquire -> npc_score_block (H2D of the slot's rows from PINNED host memory + kernels) for every "
                       "block, npc_finish (D2H of the scores).  The rows are in the pinned slots the library lends -- where a reader writes them "
                       "(the host library inflates BCF GT payloads straight into them); the timed region does not rewrite them",
               "with_host_fill": {"value": float(n) * Ve * world / dt_fill, "ms_per_step": dt_fill * 1e3, "fill_threads": T,
                                  "note": f"the same with every block first copied from pageable host memory into the slot by {T} host threads, "
                                          "inside the timed region: what a caller pays when its rows live elsewhere"}}
        assert np.isfinite(scores_host).all()
        pool.shutdown()
        e_eng.close()
        del host_gt

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r, Vc, dt = cpu_oracle_rate(n, args.cpu_seconds, 1)
        af_ms = cpu_af_test_ms_per_locus(n)
        cpu = {"value": r, "unit": "genotypes/s", "cores": 1, "kind": "port",
               "sample": f"{Vc} variants x {n} samples of the same cohort, {dt:.1f} s, single thread like the "
                         "reference; scoring only (AF-mismatch binomTest, a warning, not run)",
               "value_with_af_test": n / (dt / Vc + af_ms * 1e-3), "af_test_ms_per_locus": af_ms,
               "with_af_test_note": "the reference's default --afmisp also runs one O(n) binomTest per locus; timed on 24 loci of the sample"}

    extra = None
    if rank == 0 and world == 1 and not args.no_extra and not args.brief and args.config == 3:
        eng.close()
        del gt, d_rows
        torch.cuda.empty_cache()
        extra, _ = extra_configs(nb, torch, dev, peak)

    if rank == 0:
        line = {
            "metric": "genotypes scored/sec (variants x samples)", "value": value, "unit": "genotypes/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"config3 genome-wide PRS shard: {V} variants x {n} samples per GPU "
                                   f"(1/8 of 1M x 500k), int8 diploid BCF GT, {MISS_RATE:.1%} missing, default policies",
                       "samples": n, "variants_per_gpu": V, "block_rows": block_rows, "parallelism": f"variant-shard x{world}",
                       "kernel_shape": shape,
                       "l2": "inputs larger than L2 (shard >> 126 MB), no flush needed"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        if parity_checked is not None:
            line["parity_checked"] = parity_checked
            line["parity_note"] = (f"first {min(512, V)} rows of every rank's shard: npc_comm_combine over {world} GPUs == rank-order sum of the "
                                   "same rows scored alone on rank 0's GPU, bit for bit, nloci equal")
        if extra:
            line["extra"] = extra
        if args.brief:
            print(f"{value:.4e} genotypes/s  frac={roofline['frac']:.3f}  ms={ms_step:.3f} launch_ms={launch_ms:.3f}  {shape}")
        else:
            print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
