#!/usr/bin/env python
"""Benchmark of the LDWeaver hot path on B200: weighted SNP-pair MI/sec (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this framework (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm's CPU path (oracle port)

A "step" is one full weighted pairwise-MI scan (all make_blocks blocks: GEMM + fused MI epilogue + sr/lr link
filter + per-block exact LR selection + link-column materialisation) of the synthetic 616 x 100k alignment
(SURVEY.md 8d, config C2; --config C4 / C5 select the other scan shapes, C3 the weights-only one), blocks dealt by
cost over the ranks.  Every rank is one member of a device group (ldw_group_*, the product's multi-GPU path): rank 0
alone holds the class matrix on the host, the others receive it by NCCL broadcast; the weights come from the group
(tiles dealt + all-reduce when large enough).  `value` is pairs/s with the class matrix resident in HBM (device time
from CUDA events on the library's stream, max over ranks); `e2e` is the same metric through the C ABI from host
buffers: host->device upload (+ broadcast) + operand packing + scan + device->host copy of every link column,
inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

SR_DIST = 20000.0
LR_RETAIN = 1e6
MAX_BLK = 10000


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", help="C2 = the headline (616 x 100k); C3 = weights only (10000 x 50k); C4 = 5000 x 300k; C5 = 2000 x 500k, SNP-only chain")
    ap.add_argument("--nsnp", type=int, default=0, help="override the number of SNPs (debug only; invalidates the metric)")
    ap.add_argument("--cpu-sample", type=int, default=4000, help="block edge of the bounded CPU-baseline sample")
    ap.add_argument("--nrate", type=float, default=-1.0, help="override the per-cell N rate (debug only; invalidates the metric)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-post", action="store_true", help="skip the timing of the post-scan host steps")
    ap.add_argument("--no-extra", action="store_true", help="skip the stages reported beside the metric (wall time to links, C5 chain)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64; "
                         "link tables as a fixed, seeded sample of rows) so that two builds can be compared output for output. "
                         "The timed steps keep their link rows on the device: the rows written come from one more scan of the same "
                         "inputs, whose counts, thresholds and probabilities must equal the last timed step's")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


DUMP_ROWS = 400_000  # rows sampled per link table: 2 tables x 8 float64 columns x 400k rows = 51 MB, under 64 MB in all
LINK_COLS = ("pos1", "pos2", "clust1", "clust2", "len", "block", "MI")


def sample_rows(n: int, k: int = DUMP_ROWS) -> np.ndarray:
    """Row indices of a link table of n rows that --dump-outputs writes: all of them, or k drawn with a fixed seed (sorted)."""
    if n <= k:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def dump_outputs(out_dir: str, arrays: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d.get("hbm_gbs"), "bf16_tflops": d.get("bf16_tflops"),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  The sampler is
    started before the warm-up (nvidia-smi needs a few hundred ms to produce its first line) and only the samples whose
    timestamps fall inside the timed window are used; if the window is shorter than the sampling period the nearest
    samples (within 0.5 s, i.e. still under the same back-to-back load) are reported and flagged."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.idx)], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def window_begin(self):
        self.t0 = time.time()

    def window_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)  # let the sample that covers the end of the window land
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.strip().split(", ") for r in open(self.tmp.name) if r.strip()]
        os.unlink(self.tmp.name)
        import datetime
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        samples = []
        for r in rows:
            try:
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rs = [nm for k, nm in enumerate(names) if "Active" in r[4 + k] and "Not" not in r[4 + k]]
                samples.append((ts, float(r[1]), float(r[2]), rs))
            except Exception:
                pass
        t0, t1 = self.t0 or 0.0, self.t1 or 1e18
        inside = [s for s in samples if t0 <= s[0] <= t1]
        note = None
        if not inside:
            inside = [s for s in samples if t0 - 0.5 <= s[0] <= t1 + 0.5]
            note = f"timed window of {1e3 * (t1 - t0):.0f} ms is shorter than the sampling period: nearest samples (+-0.5 s, same back-to-back load)"
        out = {"sm_mhz": float(np.median([s[1] for s in inside])) if inside else None,
               "sm_max_mhz": max(s[2] for s in inside) if inside else None,
               "reasons": sorted({r for s in inside for r in s[3]}), "samples": len(inside)}
        if note:
            out["note"] = note
        return out


def cpu_reference_sample(codes, POS, g, hdw, edge: int, ncores: int):
    """The reference algorithm's CPU path (oracle C port, `ncores` OpenMP threads -- set explicitly, torchrun exports
    OMP_NUM_THREADS=1) on a bounded sample of the same workload: one off-diagonal `edge` x `edge` block (25 weighted
    products + temporaries + fastHadamard, pair enumeration, len, type-7 quantile, filter).  Returns (pairs, seconds)."""
    import c_oracle as CO
    n = codes.shape[0]
    edge = min(edge, n // 2)
    f = np.arange(0, edge)
    t = np.arange(n - edge, n)
    table = np.zeros((n, 5))
    for idx in (f, t):
        sub = codes[idx]
        table[idx] = np.stack([(sub == a).any(axis=1) for a in range(5)], axis=1)
    r = table.sum(axis=1)
    t0 = time.perf_counter()
    MI = CO.block_mi(codes, hdw, r, table, f, t, ncores=ncores)
    L = CO.block_links(MI, POS.astype(np.float64), f, t, float(g), SR_DIST, LR_RETAIN, 4.9e9)
    dt = time.perf_counter() - t0
    return len(L["MI"]), dt


def make_workload(cfg: str, nsnp_override: int, nrate_override: float, need_codes: bool):
    """Synthetic inputs of the BASELINE configurations (SURVEY 8d).  C2 uses the full founder / allele-frequency generator
    (as in round 1, so numbers stay comparable); the larger shapes use the uint8-only generator of the same structure
    (founders + 3 % re-draws + N), which is what fits the host's minutes.  POS / paint never depend on the codes, so ranks
    that receive the matrix by NCCL broadcast (need_codes False) skip generating it."""
    from ldweaver_b200 import synth
    S, n_cfg, seed, probs, nrate = synth.CONFIGS[cfg]
    n = nsnp_override or n_cfg
    if nrate_override >= 0:
        nrate = nrate_override
    if cfg == "C2":
        sy = synth.generate(S, n, seed, probs, nrate)
        return dict(S=S, n=n, seed=seed, codes=sy.codes, POS=sy.POS, paint=sy.paint, g=sy.g, generator="synth.generate")
    rng = np.random.default_rng(seed)
    g = synth.G_DEFAULT
    POS = np.sort(rng.choice(np.arange(1, g + 1), size=n, replace=False)).astype(np.int32)
    paint = np.ones(n, dtype=np.int32)
    paint[n // 3:] = 2
    paint[2 * n // 3:] = 3
    codes = synth.cheap_codes(S, n, seed, nrate, probs) if need_codes else None
    return dict(S=S, n=n, seed=seed, codes=codes, POS=POS, paint=paint, g=g, generator="synth.cheap_codes")


def int8_peak_tops(device):
    """cuBLASLt int8 GEMM (torch._int_mm, 8192^3, int32 accumulation) on this GPU, at this run's clocks: the measured
    denominator for the scan kernel's EXECUTED int8 tensor work.  Returns (burst TOP/s = best of 10, sustained TOP/s =
    back to back for ~1.5 s), or None when the library call is unavailable."""
    import torch
    try:
        N = 8192
        a = torch.randint(-127, 127, (N, N), dtype=torch.int8, device=device)
        b = torch.randint(-127, 127, (N, N), dtype=torch.int8, device=device)
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        reps = max(10, int(1500.0 / best))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch._int_mm(a, b)
        e1.record()
        torch.cuda.synchronize()
        sus = e0.elapsed_time(e1) / reps
        ops = 2.0 * N * N * N
        return ops / (best * 1e-3) / 1e12, ops / (sus * 1e-3) / 1e12
    except Exception:  # noqa: BLE001
        return None


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from ldweaver_b200 import synth
    ncpu = os.cpu_count() or 1

    if args.config not in ("C2", "C3", "C4", "C5"):
        raise SystemExit("--config must be one of C2 (the headline), C3 (weights only), C4, C5")
    S, n_cfg, seed, probs, nrate = synth.CONFIGS[args.config]
    n = args.nsnp or n_cfg
    workload = f"{args.config}: synthetic {S} seqs x {n} SNPs (seed {seed}), Hamming-weighted MI, sr_dist {int(SR_DIST)}, " \
               f"lr_retain_links {int(LR_RETAIN)}, max_blk_sz {MAX_BLK}"
    config = {"workload": workload, "nseq": S, "nsnp": n, "sr_dist": SR_DIST, "lr_retain_links": LR_RETAIN,
              "max_blk_sz": MAX_BLK, "partition": f"make_blocks blocks dealt by cost (pairs, largest first, least-loaded rank) over {world} rank(s)",
              "l2": "inputs larger than L2: operand planes + records exceed the 126 MB L2 and every step writes gigabytes of link columns, "
                    "so no input survives in L2 between timed steps; no explicit flush"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        import c_oracle as CO
        wl = make_workload(args.config, args.nsnp, args.nrate, True)   # the SAME data as the GPU arm
        hdw, _ = CO.hdw(wl["codes"], 0.1)
        edge = args.cpu_sample
        for _ in range(min(args.warmup, 1)):
            cpu_reference_sample(wl["codes"], wl["POS"], wl["g"], hdw, min(500, edge), ncpu)
        pairs = 0
        secs = 0.0
        for _ in range(args.steps):
            p_, dt = cpu_reference_sample(wl["codes"], wl["POS"], wl["g"], hdw, edge, ncpu)
            pairs += p_
            secs += dt
        val = pairs / secs
        sample = f"one off-diagonal {edge}x{edge} block of the same {S} x {n} workload per step (first {edge} x last {edge} SNPs; " \
                 f"reference-shaped C/OpenMP port of R/computePairwiseMI.R + src/computeMI.cpp, {ncpu} OpenMP threads set explicitly)"
        line = {"impl": "reference", "metric": "weighted SNP-pair MI/sec", "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": ncpu, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: ldweaver_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL writes its version banner / debug lines to stdout; rank 0's stdout must hold the JSON line only
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import ldweaver_b200 as ldw
    from ldweaver_b200 import api

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def finish():
        if world > 1:
            dist.destroy_process_group()
        return 0

    # Only rank 0 holds the class matrix on the host; the other ranks receive it over NVLink (ldw_group_load_codes:
    # one upload + ncclBroadcast), exactly as the product's device groups do.
    wl = make_workload(args.config, args.nsnp, args.nrate, need_codes=(rank == 0))
    POS, paint, g = wl["POS"], wl["paint"], wl["g"]
    config["generator"] = wl["generator"]
    codes_pin = torch.from_numpy(wl["codes"]).pin_memory().numpy() if rank == 0 else None
    wl["codes"] = None
    # one rank of the job's device group (world = 1: a one-member group, no NCCL)
    uid = [api.DeviceGroup.unique_id() if (rank == 0 and world > 1) else None]
    if world > 1:
        dist.broadcast_object_list(uid, src=0)
    grp = api.DeviceGroup.from_rank(local_rank, rank, world, uid[0])
    t0 = time.perf_counter()
    grp.load_codes(codes_pin, n, S)
    barrier()
    t_load = time.perf_counter() - t0
    # population-structure weights on the group: tiles of the distance GEMM dealt over the ranks + ncclAllReduce of the
    # neighbour counts when the problem is large enough (C3, C4), every rank computing all of it otherwise (C2: 616 seqs)
    grp.hdw(0.1)
    barrier()
    t0 = time.perf_counter()
    hdw, _, hdw_sharded = grp.hdw(0.1, return_parts=True)
    barrier()
    t_hdw = allmax(time.perf_counter() - t0)
    peaks = load_peaks()

    if args.config == "C3":   # weights only (BASELINE config 3): the metric of this line is the HDW stage itself
        times = []
        for _ in range(args.warmup):
            grp.hdw(0.1)
        for _ in range(args.steps):
            barrier()
            t0 = time.perf_counter()
            w_last = grp.hdw(0.1)
            barrier()
            times.append(allmax(time.perf_counter() - t0))
        if rank != 0:
            return finish()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"hdw": w_last})
        ops = 5.0 * n * S * S  # SURVEY 8d: algorithmic int8 work of the five one-hot crossprods
        i8 = int8_peak_tops(torch.device("cuda", local_rank))
        pk = i8[0] if i8 else 2 * peaks["bf16_tflops"]
        tmin = min(times)
        line = {"metric": "Hamming-distance weights: sequence pairs/sec (C3, hdw only)", "value": (S * (S - 1) / 2) / tmin, "unit": "sequence pairs/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tmin, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "int8 (tcgen05 kind::i8, int32 accumulation, exact)", "data": "synthetic", "config": config,
                "roofline": {"bound": "tensor", "achieved": ops / tmin / 1e12, "peak": pk, "unit": "TOP/s (int8)", "frac": ops / tmin / 1e12 / pk,
                             "peak_source": "torch._int_mm 8192^3 measured in this run (burst)" if i8 else "2 x MEASURED_PEAKS bf16_tflops",
                             "note": "ALGORITHMIC 5*nsnp*S^2 int8 op over the wall time of ldw_group_hdw from the device-resident matrix (allele statistics + "
                                     "plane packing + upper-triangle GEMM + count); the kernel executes ~1.3*nsnp planes over half the square",
                             "traffic": None},
                "detail": {"hdw_sharded_over_ranks": bool(hdw_sharded), "times_ms": [1e3 * t for t in times], "load_codes_s": t_load}}
        print(json.dumps(line))
        return finish()

    lra = synth.exact_lr_links_approx(POS, g, SR_DIST)
    blk = api.round_half_even_thousands(MAX_BLK)
    # C5: 2.3e9 short-range links (72 GB of columns) do not fit a host table; its long-range links are what is fed on
    base_flags = api.SCAN_LR_ONLY if args.config == "C5" else 0
    flags_dev = base_flags | api.SCAN_NO_D2H

    def scan(flags):
        return grp.mi_scan(hdw, POS, paint, blk, float(g), SR_DIST, LR_RETAIN, lra, flags, copy=False)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        scan(flags_dev)
    barrier()
    sampler.window_begin()
    t_wall0 = time.perf_counter()
    dev_ms = 0.0
    kern_ms = 0.0
    step_ms = []
    stats = None
    agg = {"n_pairs": 0, "n_launches": 0, "n_scan_launches": 0, "exec_int8_ops": 0.0, "exec_mufu_ops": 0.0, "n_tiles": 0}
    for _ in range(args.steps):
        sr_n, lr_n, _, thr_last, prob_last, st_list = scan(flags_dev)
        stats = st_list[0]
        dev_ms += stats["t_scan_ms"] + stats["t_select_ms"]
        step_ms.append(stats["t_scan_ms"] + stats["t_select_ms"])
        kern_ms += stats["t_kernel_ms"]
        for k in agg:
            agg[k] += stats[k]
    barrier()
    t_wall = time.perf_counter() - t_wall0
    sampler.window_end()
    clocks = sampler.stop()

    dev_ms_max = allmax(dev_ms)
    wall_max = allmax(t_wall)
    pairs_all = allsum(float(agg["n_pairs"]))  # over all ranks and steps
    launches_all = allsum(float(agg["n_launches"]))
    value = pairs_all / (dev_ms_max * 1e-3)

    # ------------------------------------------------------------------ end to end through the C ABI from host buffers
    e2e = None
    post = None
    sr = lr = None
    if not args.no_e2e:
        e_steps = max(1, min(args.steps, 10))
        grp.load_codes(codes_pin, n, S)   # warm-up: the pinned output tables get allocated once
        scan(base_flags)
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        pe = 0
        t_up = t_scan = 0.0
        for _ in range(e_steps):
            ta = time.perf_counter()
            grp.load_codes(codes_pin, n, S)            # host -> device (rank 0) + NCCL broadcast
            tb = time.perf_counter()
            sr, lr, bd, thr, prob, st2 = scan(base_flags)  # operand packing + scan + device -> host copy of every link column
            tc = time.perf_counter()
            d2h += (int(sr.n) + int(lr.n)) * 32
            pe += st2[0]["n_pairs"]
            t_up += tb - ta
            t_scan += tc - tb
        barrier()
        te = allmax(time.perf_counter() - t0)
        st2 = st2[0]
        # what follows the scan in perform_MI_computation (R/computePairwiseMI.R:118-143), native host code, on the
        # short-range table the last step left in pinned host memory: reported beside the metric, not part of it
        if rank == 0 and world == 1 and not args.no_post and args.config == "C2":
            try:
                tp0 = time.perf_counter()
                sp = api.mergeNsort_sr_links(ldw.CdsVar(paint, 3), sr, SR_DIST, None, 3.0)
                tp1 = time.perf_counter()
                ar = api.runARACNE({k: sp.df[k][sp.red] for k in ("pos1", "pos2", "MI")}, {k: sp.df[k][sp.chk] for k in ("pos1", "pos2", "MI")})
                tp2 = time.perf_counter()
                post = {"mergeNsort_sr_links_s": tp1 - tp0, "runARACNE_s": tp2 - tp1, "n_sr_links": int(sr.n), "n_df": int(len(sp.df["row"])),
                        "n_red": int(len(sp.red)), "n_aracne_check": int(len(sp.chk)), "aracne_kept": int(ar.sum()),
                        "beta_shapes": [f["shape"].tolist() for f in sp.fits], "nm_evals": [f["nm_evals"] for f in sp.fits],
                        "host_threads": ncpu}
            except Exception as ex:  # noqa: BLE001 -- a failed fit must not take the metric down with it
                post = {"error": str(ex)}
        pe_all = allsum(float(pe))
        d2h_all = allsum(float(d2h))
        h2d = (n * S if rank == 0 else 0) + hdw.nbytes + POS.nbytes + paint.nbytes
        h2d_all = allsum(float(h2d))
        e2e = {"value": pe_all / te, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all // e_steps),
               "ms_per_step": 1e3 * te / e_steps, "steps": e_steps,
               "breakdown_ms": {"load_codes (H2D on rank 0 + ncclBroadcast)": 1e3 * t_up / e_steps, "group_mi_scan call": 1e3 * t_scan / e_steps,
                                "operand packing (inside the call)": st2["t_plan_ms"], "scan_device": st2["t_scan_ms"] + st2["t_select_ms"],
                                "scan_kernels": st2["t_kernel_ms"], "select_tail": st2["t_select_ms"], "host_prep": st2["t_host_prep_ms"], "d2h_tail": st2["t_d2h_ms"]},
               "includes": "host->device upload of the class matrix (rank 0) and its NCCL broadcast, operand packing on every rank, scan, link "
                           "materialisation, device->host copy of all link columns into pinned host memory"
                           + (" (C5: long-range links only, LDW_SCAN_LR_ONLY)" if args.config == "C5" else "")}

    # ------------------------------------------------------------------ beside the metric (rank 0, one GPU): the other stages
    extra = {}
    if rank == 0 and world == 1 and not args.no_extra:
        try:
            if args.config == "C5" and lr is not None:
                # BASELINE config 5 as stated: SNP-only input through the encoder (relaxed filter), then the long-range links
                # of the scan into analyse_long_range_links -> runARACNE
                aln = synth.codes_to_alignment(codes_pin, lowercase_frac=0.3)
                t0 = time.perf_counter()
                snp5 = ldw.snp_dat_from_alignment_matrix(aln, pos=POS, method="relaxed", device=local_rank)
                t_enc = time.perf_counter() - t0
                del aln
                lrd = lr.to_dict()
                t0 = time.perf_counter()
                empty = {k: np.zeros(0) for k in ("pos1", "pos2", "MI")}
                lr_red = api.analyse_long_range_links({"pos1": lrd["pos1"].astype(float), "pos2": lrd["pos2"].astype(float), "c1": lrd["clust1"],
                                                       "c2": lrd["clust2"], "len": lrd["len"].astype(float), "MI": lrd["MI"]}, empty)
                t_ar = time.perf_counter() - t0
                extra["C5_chain"] = {"encode_relaxed_s": t_enc, "nsnp_retained": int(snp5.nsnp),
                                     "codes_identical_to_generator": bool(snp5.nsnp == n and np.array_equal(snp5.codes, codes_pin)),
                                     "n_lr_links": int(len(lrd["MI"])), "analyse_long_range_links_s": t_ar, "n_lr_links_red": int(len(lr_red["MI"])),
                                     "aracne_kept": int(np.sum(lr_red["ARACNE"])),
                                     "note": "ARACNE check set = long-range links above the Tukey threshold (the short-range table is not materialised at this size)"}
            if args.config == "C2":
                # wall time "to sr/lr links" through the public API (the metric's second half): hdw + perform_MI_computation with both TSVs
                snp = ldw.snp_dat_from_codes(codes_pin, POS, g)
                with tempfile.TemporaryDirectory() as d:
                    for variant, kw in (("host_post", dict(exact_sr="in_scan")), ("device_post", dict(device_post=True))):
                        for it in range(2):  # second call reported (the first allocates pinned buffers)
                            for f in ("lr_links.tsv", "sr_links.tsv"):
                                if os.path.exists(os.path.join(d, f)):
                                    os.unlink(os.path.join(d, f))
                            t0 = time.perf_counter()
                            h2 = ldw.estimate_Hamming_distance_weights(snp, 0.1, device=local_rank)
                            t1 = time.perf_counter()
                            res = ldw.perform_MI_computation(snp, h2, ldw.CdsVar(paint, 3), ncores=1, lr_save_path=os.path.join(d, "lr_links.tsv"),
                                                             sr_save_path=os.path.join(d, "sr_links.tsv"), plt_folder=d, sr_dist=SR_DIST, lr_retain_links=LR_RETAIN,
                                                             max_blk_sz=MAX_BLK, srp_cutoff=3, runARACNE=True, lr_links_approx=lra, device=local_rank, **kw)
                            t2 = time.perf_counter()
                        extra["wall_to_links_" + variant] = {
                            "total_s": t2 - t0, "hdw_s": t1 - t0, "perform_MI_computation_s": t2 - t1, "n_sr_links": int(res.stats["n_sr"]),
                            "n_lr_links": int(len(res.lr["MI"])), "n_sr_links_red": int(len(res.sr_links_red["row"])), "phases_s": res.stats.get("phases"),
                            "short_range_MI": "fp64, recomputed inside the scan (LDW_SCAN_SR_EXACT)",
                            "includes": "hdw + upload/packing + scan + lr_links.tsv + mergeNsort_sr_links + runARACNE + ordering + sr_links.tsv"
                                        + (" + D2H of the whole short-range table and its NumPy copies; mergeNsort_sr_links on host threads" if variant == "host_post"
                                           else "; short-range table kept in device memory, mergeNsort_sr_links on the device (ldw_sr_postprocess_dev)"),
                            "host_threads": ncpu}
                    extra["wall_to_links_s"] = extra["wall_to_links_device_post"]["total_s"]
                    del res
        except Exception as ex:  # noqa: BLE001
            extra["error"] = repr(ex)

    if args.dump_outputs:
        # The timed steps leave their link columns in device memory (LDW_SCAN_NO_D2H).  One more scan of the same inputs
        # copies them out; the scan is deterministic, and its counts, thresholds and probabilities must equal the last
        # timed step's before its rows are written as that step's.
        sr_d, lr_d, _, thr_d, prob_d, _ = scan(base_flags)
        if rank == 0:
            if (int(sr_d.n), int(lr_d.n)) != (int(sr_n.n), int(lr_n.n)) or not (
                    np.array_equal(thr_d, thr_last, equal_nan=True) and np.array_equal(prob_d, prob_last, equal_nan=True)):
                raise SystemExit("--dump-outputs: a repeated scan of the same inputs differs from the last timed step")
            out = {"thr": thr_last, "prob": prob_last, "n_links": np.array([int(sr_n.n), int(lr_n.n)])}
            for tag, tbl in (("sr", sr_d), ("lr", lr_d)):
                rows = sample_rows(int(tbl.n))
                cols = tbl.views()
                if rows.size and set(LINK_COLS) - set(cols):
                    raise SystemExit(f"--dump-outputs: {tag} link table lacks columns {sorted(set(LINK_COLS) - set(cols))}")
                out[f"{tag}_rows"] = rows
                for k in LINK_COLS:
                    out[f"{tag}_{k}"] = cols[k][rows] if rows.size else np.zeros(0)
            dump_outputs(args.dump_outputs, out)

    if rank != 0:
        return finish()

    # ------------------------------------------------------------------ roofline of the dominant kernel (mi_scan_kernel)
    n_launch = max(1, agg["n_scan_launches"])
    avg_launch_s = kern_ms * 1e-3 / n_launch
    alg_flop_per_launch = 50.0 * S * (agg["n_pairs"] / n_launch)  # SURVEY.md 8d: 50*S flop per SNP pair
    alg_tf = alg_flop_per_launch / avg_launch_s / 1e12
    exec_tops = agg["exec_int8_ops"] / (kern_ms * 1e-3) / 1e12
    i8 = int8_peak_tops(torch.device("cuda", local_rank)) if world == 1 else None
    i8_peak = i8[0] if i8 else 2.0 * peaks["bf16_tflops"]
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    num_sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    mufu_peak = 16.0 * num_sms * sm_mhz * 1e6      # 16 MUFU results / clk / SM (4 per scheduler)
    mufu_rate = agg["exec_mufu_ops"] / (kern_ms * 1e-3)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "mi_scan_traffic.json")
    if os.path.exists(tpath) and args.config == "C2" and not args.nsnp:
        tj = json.load(open(tpath))
        traffic = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]  # from one ncu --set full capture
    bf16_pk = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
    roofline = {"bound": "tensor", "achieved": exec_tops, "peak": i8_peak, "unit": "TOP/s (int8)", "frac": exec_tops / i8_peak,
                "traffic": traffic,
                "peak_source": ("cuBLASLt int8 GEMM (torch._int_mm 8192^3, int32 accumulate) measured in this run on this GPU: burst %.0f, sustained %.0f TOP/s"
                                % (i8[0], i8[1])) if i8 else "2 x MEASURED_PEAKS.json bf16_tflops (int8 microbenchmark not run at N > 1)",
                "nominal_peak": 4500.0, "frac_of_nominal": exec_tops / 4500.0,
                "peak_note": "the library GEMM does not reach the nominal dense int8 rate (4.5 POP/s) on this pool; when this kernel's tensor work "
                             "runs faster than it (5000-sequence shapes) frac exceeds 1 and frac_of_nominal is the figure to read",
                "kernel": "mi_scan_kernel", "avg_launch_ms": 1e3 * avg_launch_s, "launches": n_launch,
                "kernel_share_of_step": kern_ms / dev_ms if dev_ms else None,
                "what": "EXECUTED int8 tensor op/s of the scan kernel (2 x MACs of every cta_group::2 UMMA it issues, M = 256: (r_i-1)(r_j-1) plane "
                        "pairs x 2 weight halves x 2 digit passes, halves of a pair tile without wanted pairs included) over its CUDA-event time, "
                        "against the measured int8 peak",
                "mufu": {"executed_per_s": mufu_rate, "peak_per_s": mufu_peak, "frac": mufu_rate / mufu_peak,
                         "what": "MUFU.LG2 / MUFU.RCP lane-results of the epilogue (counted per tile kind from the kernel's term loop) against "
                                 "16 / clk / SM x %d SMs at the sampled %.0f MHz" % (num_sms, sm_mhz)},
                "algorithmic": {"achieved_tflops": alg_tf, "peak_tflops": bf16_pk, "frac": alg_tf / bf16_pk,
                                "what": "SURVEY 8d: 50*S flop per SNP pair (all 25 weighted dot products in one bf16 pass) over the same time, against "
                                        "MEASURED_PEAKS.json bf16_tflops_sustained (%s); exceeds 1 because only r-1 planes per site enter the int8 GEMM" % peaks["source"]}}

    cpu = None
    if not args.no_cpu and world == 1:
        pr, dt = cpu_reference_sample(codes_pin, POS, g, hdw, args.cpu_sample, ncpu)
        e_ = min(args.cpu_sample, n // 2)
        cpu = {"value": pr / dt, "unit": "pairs/s", "cores": ncpu, "kind": "port",
               "sample": f"one off-diagonal {e_}x{e_} block of the same workload ({pr} pairs, {dt:.1f} s), reference-shaped C/OpenMP port of "
                         f"R/computePairwiseMI.R + src/computeMI.cpp, {ncpu} OpenMP threads"}

    line = {"metric": "weighted SNP-pair MI/sec", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int8 (tcgen05 kind::i8 with int32 accumulation of 28-bit fixed-point weights; fp32 MI epilogue, fp64 refinement of long-range links)",
            "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_all),
            "roofline": roofline, "cpu_baseline": cpu,
            "detail": {"wall_ms_per_step": 1e3 * wall_max / args.steps, "post_scan_host": post,
                       "wall_to_links_s": extra.get("wall_to_links_s"), "extra": extra,
                       "step_ms": {"min": min(step_ms), "median": sorted(step_ms)[len(step_ms) // 2], "max": max(step_ms)},
                       "hdw_s": t_hdw, "hdw_sharded_over_ranks": bool(hdw_sharded), "load_codes_s": t_load,
                       "pack_ms": stats["t_pack_ms"], "host_prep_ms": stats["t_host_prep_ms"],
                       "pairs_per_step": pairs_all / args.steps, "n_sr": stats["n_sr"], "n_lr_kept": stats["n_lr_kept"],
                       "n_reruns": stats["n_reruns"], "n_candidates": stats["n_candidates"], "tiles_per_step_rank0": agg["n_tiles"] / args.steps,
                       "lr_links_approx": lra}}
    print(json.dumps(line))
    return finish()


if __name__ == "__main__":
    sys.exit(main())
