#!/usr/bin/env python
"""bench.py - KING N x N pair-dot-products/s on the BASELINE.json workload (100k samples x 1M SNPs).

A "step" is one pass of the hot path (the KING pair-count kernel, CalcKing's dense loop) over one
batch of `--batch-variants` synthetic variants for ALL sample pairs of this rank's row block; the
counts accumulate in HBM across steps exactly as in a full run (8 steps of 131,072 variants = one
1M-SNP job).

  value   = (pairs x variants_per_step / 1e6) / step time: full-length (1M-SNP) pair-dot-products per
            second, whole job over all ranks, inputs already resident in HBM.
  e2e     = same metric through the C-ABI with HOST buffers: every step copies the step's genotype
            batch (1/G of it per rank) from pinned host memory and reads back 1/steps_per_job of the
            fp64 kinship matrix.
  roofline= int8 tensor pipe: 5 products x 2 ops x pairs x variants / tensor-kernel time (CUDA events
            recorded by the library around the launch, on the stream it is launched on) vs the int8 rate
            MEASURED on this GPU in the same run (pl2gpu_int8_peak: tcgen05.mma kind::i8 on all SMs
            for >= 2 s).
  cpu_baseline / --impl reference = the UNMODIFIED reference binary (oracle/_ref/plink2,
            --make-king-table, as many threads as this process may actually use) on a bounded sample.

Multi-GPU (torchrun, one rank per GPU): rows of the output triangle are split into tile-aligned
equal-work blocks; each rank holds 1/G of the step's variants and the LIBRARY (NCCL inside
libpl2gpu, pl2gpu_king_add_variants_sharded) all-gathers the genotype column tile on its prep stream,
double-buffered against the previous step's tensor kernel; outputs stay local.  Total work is fixed
=> "strong" scaling.
"""
import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FULL_N = 100_000
FULL_M = 1_000_000
METRIC = "KING NxN pair-dot-products/sec (100k samples x 1M SNPs)"
UNIT = "pair-dot-products/s (1M-SNP pairs)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples", type=int, default=FULL_N)
    ap.add_argument("--batch-variants", type=int, default=131072)
    ap.add_argument("--algo", default="tensor_ts", choices=["tensor_ts", "tensor", "popcount"])
    ap.add_argument("--row-split", default="tiles", choices=["tiles", "parallel"], help="multi-GPU row blocks: tile-aligned equal work, or the reference's ParallelBounds")
    ap.add_argument("--cpu-samples", type=int, default=16384)
    ap.add_argument("--cpu-variants", type=int, default=65536)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short GRM / PCA / LD measurements reported under `secondary`")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of the KING pairs (counts and kinship) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ----------------------------------------------------------------------------------- synthetic data
def synth_genovecs(torch, n, v0, v1, device, seed=20260923, miss=0.01):
    """uint8 [v1-v0, 8*ceil(n/32)] PgrGet-layout rows: HWE genotypes, per-variant ALT freq ~U(.02,.98),
    1% missing (the shape of the reference's --dummy generator, 2.0/plink2_import.cc:16326-16460).
    Deterministic in (seed, variant index) so every rank can synthesise its own slice."""
    row_bytes = (n + 31) // 32 * 8
    out = torch.empty((v1 - v0, row_bytes), dtype=torch.uint8, device=device)
    n4 = row_bytes * 4
    chunk = max(1, min(v1 - v0, (1 << 28) // max(n4, 1)))
    for s in range(v0, v1, chunk):
        e = min(v1, s + chunk)
        g = torch.Generator(device=device)
        g.manual_seed(seed * 1_000_003 + s)
        f = torch.rand((e - s, 1), generator=g, device=device) * 0.96 + 0.02
        code = (torch.rand((e - s, n4), generator=g, device=device) < f).to(torch.uint8)
        code += (torch.rand((e - s, n4), generator=g, device=device) < f).to(torch.uint8)
        code[torch.rand((e - s, n4), generator=g, device=device) < miss] = 3
        if n4 > n:
            code[:, n:] = 0
        q = code.view(e - s, row_bytes, 4)
        out[s - v0 : e - v0] = q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)
        del code, q, f
    return out


# --------------------------------------------------------------------------------------- host CPUs
def effective_cores():
    """What this process may actually run on: the affinity mask capped by the cgroup CPU quota (round 1
    reported os.cpu_count() = 128 on a lease that behaved like ~1/5 of that)."""
    aff = len(os.sched_getaffinity(0))
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    used = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return {"os_cpu_count": os.cpu_count(), "affinity": aff, "cgroup_quota_cpus": quota, "threads_used": used}


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------- reference CPU arm
def write_synth_bed(prefix, n, m):
    """n x m synthetic .bed/.bim/.fam (same generator as the GPU steps); variant k sits at bp k+1 of chr 1."""
    import torch

    dev = "cuda" if torch.cuda.is_available() else "cpu"
    # PgrGet codes -> .bed codes (0 homALT,1 missing,2 het,3 homREF; pgen_spec.tex:436-438)
    lut = torch.tensor([3, 2, 0, 1], dtype=torch.uint8, device=dev)
    bpv = (n + 3) // 4
    with open(prefix + ".bed", "wb") as f:
        f.write(bytes([0x6C, 0x1B, 0x01]))
        for s0 in range(0, m, 2048):
            s1 = min(m, s0 + 2048)
            by = synth_genovecs(torch, n, s0, s1, dev)[:, :bpv].contiguous()
            c = torch.stack([(by >> sh) & 3 for sh in (0, 2, 4, 6)], dim=-1).to(torch.int32)
            b = lut[c]
            if n % 4:
                b.view(s1 - s0, -1)[:, n:] = 0
            bed = (b[..., 0] | (b[..., 1] << 2) | (b[..., 2] << 4) | (b[..., 3] << 6)).to(torch.uint8).cpu().numpy()
            bed.tofile(f)
            del by, c, b, bed
    with open(prefix + ".bim", "w") as f:
        f.write("".join(f"1\tsnp{k}\t0\t{k + 1}\tA\tG\n" for k in range(m)))
    with open(prefix + ".fam", "w") as f:
        f.write("".join(f"0\tper{k}\t0\t0\t2\t-9\n" for k in range(n)))


def run_cli(binary, prefix, out, flags, threads=None):
    cmd = [binary, "--bfile", prefix] + flags + ["--out", out]
    if threads is not None:
        cmd += ["--threads", str(threads), "--memory", "64000"]
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError(os.path.basename(binary) + " failed: " + r.stdout[-500:] + r.stderr[-500:])
    return dt


def ref_binary():
    plink2 = os.path.join(ROOT, "oracle", "_ref", "plink2")
    if not os.path.exists(plink2):
        raise FileNotFoundError(f"{plink2} missing (oracle/build_ref.sh builds it where /root/reference exists)")
    return plink2


def run_reference_sample(n, m, threads, workdir, keep_input=None):
    """Times the unmodified reference binary on an n x m synthetic .bed: `--make-king-table` with a
    table filter so the text output stays small (the N^2 M/64 popcount loop is unaffected).
    Returns (seconds, pair_snp_per_s, input prefix)."""
    prefix = keep_input or os.path.join(workdir, f"cpu_{n}_{m}")
    if not os.path.exists(prefix + ".bed"):
        write_synth_bed(prefix, n, m)
    dt = run_cli(ref_binary(), prefix, prefix + "_out", ["--make-king-table", "--king-table-filter", "0.35"], threads)
    pairs = n * (n - 1) // 2
    return dt, pairs * m / dt, prefix


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = effective_cores()
    threads = cores["threads_used"]
    n, m = args.cpu_samples, args.cpu_variants
    tmp = tempfile.mkdtemp(prefix="pl2ref_")
    try:
        times = []
        for it in range(args.warmup + args.steps):
            dt, _, _ = run_reference_sample(n, m, threads, tmp, keep_input=os.path.join(tmp, "in"))
            if it >= args.warmup:
                times.append(dt)
        t = sum(times) / len(times)
        pairs = n * (n - 1) // 2
        val = pairs * m / 1e6 / t
        line = {
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64 popcount (AVX2)", "data": "synthetic",
            "config": {"workload": "plink2 --make-king-table, bounded sample of the 100k x 1M job", "samples": n, "variants": m, "threads": threads, "host_cpus": cores, "pair_snp_per_s": pairs * m / t},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "host_cpus": cores, "kind": "reference", "sample": f"{n} samples x {m} variants, whole `plink2 --make-king-table --threads {threads}` run incl. .bed load"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        emit(line)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def cpu_legs(args):
    """Rank 0, N = 1: (a) cpu_baseline = the reference binary on the bounded sample, with the load phase
    separated by timing half the variants as well; (b) cli_same_files = the SAME command line through the
    reference and through plink2_b200 on the same files, a non-empty filtered table (>= 1e5 rows) and the whole
    fp32 kinship triangle compared byte for byte."""
    import numpy as np

    cores = effective_cores()
    threads = cores["threads_used"]
    n, m = args.cpu_samples, args.cpu_variants
    tmp = tempfile.mkdtemp(prefix="pl2cpu_")
    cpu_baseline, cli = None, None
    try:
        dt, rate, prefix = run_reference_sample(n, m, threads, tmp)
        pairs = n * (n - 1) // 2
        # same run on the first half of the variants: the difference is pure pair-count time (no start-up, no load of the other half)
        dt_half = run_cli(ref_binary(), prefix, prefix + "_half", ["--chr", "1", "--from-bp", "1", "--to-bp", str(m // 2), "--make-king-table", "--king-table-filter", "0.35"], threads)
        kernel_rate = pairs * (m - m // 2) / max(dt - dt_half, 1e-9) if dt > dt_half else None
        cpu_baseline = {"value": rate / 1e6, "unit": UNIT, "cores": threads, "host_cpus": cores, "kind": "reference", "seconds": dt, "seconds_half_variants": dt_half,
                        "pair_snp_per_s": rate, "pair_snp_per_s_kernel_phase": kernel_rate,
                        "sample": f"{n} samples x {m} variants, one whole `plink2 --make-king-table --threads {threads}` run (incl. .bed load) of oracle/_ref/plink2; kernel phase = difference to the same run on half the variants"}
        try:
            ours = os.path.join(ROOT, "plink_ng_b200", "plink2_b200")
            pre_ours, pre_ref = prefix + "_b200", prefix + "_ref"
            # pick the table filter from the data so that ~2e5 rows survive (unrelated samples: a fixed 0.35 keeps nothing)
            run_cli(ours, prefix, pre_ours + "_q", ["--make-king", "bin4", "triangle"])
            kin = np.fromfile(pre_ours + "_q.king.bin", dtype=np.float32)
            thr = repr(float(np.partition(kin, kin.size - 200_000)[kin.size - 200_000]))
            del kin
            flags = ["--make-king", "bin4", "triangle", "--make-king-table", "counts", "cols=+ibs1,+ibs", "--king-table-filter", thr]
            dt_ref = run_cli(ref_binary(), prefix, pre_ref, flags, threads)
            dt_ours = run_cli(ours, prefix, pre_ours, flags)
            rows = sum(1 for _ in open(pre_ref + ".kin0")) - 1
            same_tab = open(pre_ref + ".kin0", "rb").read() == open(pre_ours + ".kin0", "rb").read()
            same_mat = open(pre_ref + ".king.bin", "rb").read() == open(pre_ours + ".king.bin", "rb").read()
            cli = {"seconds_reference": dt_ref, "seconds": dt_ours, "value": pairs * m / dt_ours / 1e6, "unit": UNIT, "speedup_vs_reference_run": dt_ref / dt_ours,
                   "kin0_rows": rows, "kin0_identical_to_reference": bool(same_tab and rows >= 100_000), "king_bin_identical_to_reference": bool(same_mat),
                   "command": f"--bfile <same {n} x {m} files> {' '.join(flags)} (process start to exit: CUDA init, .bed load, H2D, kernels, matrix + table write)"}
        except Exception as ex:
            cli = {"error": str(ex)[-300:]}
    except Exception as ex:  # the baseline is reported, never silently faked
        cpu_baseline = {"value": None, "unit": UNIT, "cores": threads, "host_cpus": cores, "kind": "reference", "sample": f"unavailable: {ex}"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return cpu_baseline, cli


def hbm_peak_gbs():
    """Measured HBM copy bandwidth of this pool's B200s (driver-written MEASURED_PEAKS.json), else the profiling
    guide's fallback."""
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6500.0


# ------------------------------------------------------------------------------------- secondary
def secondary_legs(args, torch, p, ctx, dev, peak_tops):
    """Short measurements of the other kernels of the path (not the headline metric), inputs resident."""
    import numpy as np

    from plink_ng_b200.host import GrmJob

    sec = {}
    n2, m2 = min(args.samples, 16384), 65536
    try:
        g2 = synth_genovecs(torch, n2, 0, m2, dev)
        torch.cuda.synchronize()
        rf = np.random.default_rng(0).uniform(0.05, 0.95, size=m2)
        with GrmJob(ctx, n2) as gj:
            gj.add_variants_device(g2.data_ptr(), g2.shape[1], m2, ref_freqs=rf)
            ctx.synchronize()
            ctx.event_record(6)
            for _ in range(3):
                gj.add_variants_device(g2.data_ptr(), g2.shape[1], m2, ref_freqs=rf)
            ctx.event_record(7)
            g_ms = ctx.event_elapsed_ms(6, 7) / 3
        tri = n2 * (n2 + 1) // 2
        tops = 11 * 2 * tri * m2 / (g_ms * 1e-3) / 1e12
        sec["grm"] = {"kernel": "grm_ts_kernel", "workload": f"{n2} samples x {m2} variants per add_variants call (tables + re-tiling + tensor kernel), inputs resident",
                      "ms_per_call": g_ms, "achieved": tops, "unit": "TOP/s (int8; 10 digit planes + obs = 11 products x 2 ops per pair and variant)",
                      "peak": peak_tops, "frac": tops / peak_tops if peak_tops else None, "frac_of_nominal_4500": tops / 4500.0, "pair_snp_per_s": tri * m2 / (g_ms * 1e-3)}
        del g2
    except Exception as ex:  # reported, never faked
        sec["grm"] = {"error": str(ex)[-300:]}
    # CPU GRM beside it: the LAPACK build of the reference (threaded OpenBLAS dsyrk), bounded sample
    try:
        lap = os.path.join(ROOT, "oracle", "_ref", "plink2_lapack")
        if os.path.exists(lap) and "grm" in sec and "error" not in sec["grm"]:
            nc, mc = 8192, 32768
            tmp = tempfile.mkdtemp(prefix="pl2grm_")
            try:
                prefix = os.path.join(tmp, "g")
                write_synth_bed(prefix, nc, mc)
                threads = effective_cores()["threads_used"]
                dt = run_cli(lap, prefix, prefix + "_out", ["--make-grm-bin"], threads)
                sec["grm"]["cpu_baseline"] = {"kind": "reference", "binary": "oracle/_ref/plink2_lapack (OpenBLAS dsyrk, fp64)", "cores": threads, "seconds": dt,
                                              "sample": f"{nc} samples x {mc} variants, whole `--make-grm-bin` run", "pair_snp_per_s": nc * (nc + 1) // 2 * mc / dt}
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
    except Exception as ex:
        sec["grm"]["cpu_baseline"] = {"error": str(ex)[-200:]}
    # --pca approx (randomized range finder over the resident 2-bit matrix): the library call the host program makes
    try:
        import ctypes as C

        from plink_ng_b200.capi import check, lib

        n3, m3, k3 = min(args.samples, 16384), 65536, 20
        g3 = synth_genovecs(torch, n3, 0, m3, dev)
        g1 = np.random.default_rng(1).standard_normal((n3, 2 * k3))
        h = C.c_void_p()
        check(lib.pl2gpu_pca_begin(ctx.handle, n3, m3, k3, C.byref(h)), "pl2gpu_pca_begin")
        try:
            check(lib.pl2gpu_pca_add_variants(h, C.c_void_p(g3.data_ptr()), g3.shape[1], m3, 1, None), "pl2gpu_pca_add_variants")
            vals, vecs = np.empty(k3), np.empty((k3, n3))
            ctx.synchronize()
            t0 = time.perf_counter()
            check(lib.pl2gpu_pca_run(h, g1.ctypes.data, vals.ctypes.data, vecs.ctypes.data), "pl2gpu_pca_run")
            dt = time.perf_counter() - t0
        finally:
            lib.pl2gpu_pca_end(h)
        col_products = 2 * k3 * (3 * k3 + 2)  # (k+1) x 2k XA columns + k x 2k and 2k(k+1) XtB columns
        sec["pca"] = {"workload": f"--pca {k3} approx core (pl2gpu_pca_run: {k3 + 1} Y.G passes, {k3} Yt.H passes, Krylov SVD, Yt.Q, final SVD) on {n3} samples x {m3} variants, genotypes resident",
                      "seconds": dt, "fma_equiv_per_s": n3 * m3 * col_products / dt, "column_products": col_products, "top_eigenvalue": float(vals[0])}
        del g3
    except Exception as ex:
        sec["pca"] = {"error": str(ex)[-300:]}
    try:
        lap = os.path.join(ROOT, "oracle", "_ref", "plink2_lapack")
        if os.path.exists(lap) and "pca" in sec and "error" not in sec["pca"]:
            nc, mc = 8192, 32768
            tmp = tempfile.mkdtemp(prefix="pl2pca_")
            try:
                prefix = os.path.join(tmp, "g")
                write_synth_bed(prefix, nc, mc)
                threads = effective_cores()["threads_used"]
                dt = run_cli(lap, prefix, prefix + "_out", ["--pca", "20", "approx"], threads)
                sec["pca"]["cpu_baseline"] = {"kind": "reference", "binary": "oracle/_ref/plink2_lapack (OpenBLAS)", "cores": threads, "seconds": dt,
                                              "sample": f"{nc} samples x {mc} variants, whole `--pca 20 approx` run", "fma_equiv_per_s": nc * mc * 2 * 20 * 62 / dt}
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
    except Exception as ex:
        sec["pca"]["cpu_baseline"] = {"error": str(ex)[-200:]}
    # --indep-pairwise pair decisions (ld_ts_kernel) at config 4's founder count, and --score accumulation; each with the
    # reference's own command timed on a bounded sample of the same generator's data
    try:
        import ctypes as C

        from plink_ng_b200.capi import check, lib

        nf, mv, window = min(args.samples, 50000), 131072, 500
        g4 = synth_genovecs(torch, nf, 0, mv, dev)
        band = window - 1
        flags_t = torch.zeros((mv, band), dtype=torch.uint8).pin_memory()
        dt = float("inf")
        flags_ptr = flags_t.numpy().ctypes.data
        for _ in range(3):
            ctx.synchronize()
            t0 = time.perf_counter()
            check(lib.pl2gpu_ld_band_flags(ctx.handle, C.c_void_p(g4.data_ptr()), g4.shape[1], nf, mv, 1, band, 0.2 * (1 + 2.0 ** -44), flags_ptr), "pl2gpu_ld_band_flags")
            dt = min(dt, time.perf_counter() - t0)
        pairs = mv * band - band * (band + 1) // 2
        sec["ld"] = {"kernel": "ld_ts_kernel", "workload": f"pair decisions of --indep-pairwise {window} on {nf} founders x {mv} variants (whole pl2gpu_ld_band_flags call incl. staging and {flags_t.numel() / 1e6:.0f} MB of decisions to pinned host memory)",
                     "seconds": dt, "pairs_per_s": pairs / dt, "achieved": 12 * pairs * nf / dt / 1e12, "unit": "TOP/s (int8; 6 products x 2 ops per pair and founder)", "peak": peak_tops,
                     "frac": (12 * pairs * nf / dt / 1e12) / peak_tops if peak_tops else None}
        del g4, flags_t
        ref = os.path.join(ROOT, "oracle", "_ref", "plink2")
        if os.path.exists(ref):
            nc, mc = 8192, 32768
            tmp = tempfile.mkdtemp(prefix="pl2ld_")
            try:
                prefix = os.path.join(tmp, "g")
                write_synth_bed(prefix, nc, mc)
                threads = effective_cores()["threads_used"]
                dt_ref = run_cli(ref, prefix, prefix + "_out", ["--indep-pairwise", str(window), "50", "0.2"], threads)
                # the reference evaluates (almost) every pair of a window on unlinked data: variants x (window - 1 + step) / 2 ... bounded above by variants x band
                sec["ld"]["cpu_baseline"] = {"kind": "reference", "cores": threads, "seconds": dt_ref, "sample": f"{nc} founders x {mc} variants on one chromosome (one compute thread per chromosome in the reference), whole `--indep-pairwise {window} 50 0.2` run",
                                             "founder_pairs_per_s_upper_bound": nc * (mc * band) / dt_ref}
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
    except Exception as ex:
        sec.setdefault("ld", {})["error"] = str(ex)[-300:]
    try:
        import ctypes as C

        from plink_ng_b200.capi import check, lib

        ns, ms = args.samples, 131072
        g5 = synth_genovecs(torch, ns, 0, ms, dev)
        w4 = np.random.default_rng(2).normal(size=(ms, 4))
        d4 = np.full(ms, 0 | (1 << 2) | (2 << 4), dtype=np.uint8)
        h = C.c_void_p()
        check(lib.pl2gpu_score_begin(ctx.handle, ns, C.byref(h)), "pl2gpu_score_begin")
        try:
            for _ in range(2):
                ctx.synchronize()
                t0 = time.perf_counter()
                check(lib.pl2gpu_score_add_variants(h, C.c_void_p(g5.data_ptr()), g5.shape[1], ms, 1, w4.ctypes.data, d4.ctypes.data), "pl2gpu_score_add_variants")
                dt = time.perf_counter() - t0
        finally:
            lib.pl2gpu_score_end(h)
        sec["score"] = {"kernel": "score_kernel", "workload": f"--score accumulation, {ns} samples x {ms} scored entries, genotypes resident (whole pl2gpu_score_add_variants call)", "seconds": dt,
                        "sample_entries_per_s": ns * ms / dt, "achieved": ns * ms / 4 / dt / 1e9, "unit": "GB/s of 2-bit genotypes", "peak": hbm_peak_gbs(), "bound": "ALU (fp64 table add per sample and entry), then HBM"}
        del g5
        ref = os.path.join(ROOT, "oracle", "_ref", "plink2")
        if os.path.exists(ref):
            nc, mc = 8192, 65536
            tmp = tempfile.mkdtemp(prefix="pl2sc_")
            try:
                prefix = os.path.join(tmp, "g")
                write_synth_bed(prefix, nc, mc)
                with open(prefix + ".bim") as f, open(prefix + ".score", "w") as o:
                    for k, ln in enumerate(f):
                        t = ln.split()
                        o.write(f"{t[1]}\t{t[4]}\t{(k % 7 - 3) * 0.01}\n")
                threads = effective_cores()["threads_used"]
                dt_ref = run_cli(ref, prefix, prefix + "_out", ["--score", prefix + ".score"], threads)
                sec["score"]["cpu_baseline"] = {"kind": "reference", "cores": threads, "seconds": dt_ref, "sample": f"{nc} samples x {mc} scored variants, whole `--score` run", "sample_entries_per_s": nc * mc / dt_ref}
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
    except Exception as ex:
        sec.setdefault("score", {})["error"] = str(ex)[-300:]
    return sec


# ------------------------------------------------------------------------------------- outputs
DUMP_ROWS, DUMP_COLS = 64, 4096


def dump_outputs(job, r0, r1, out_dir):
    """What a caller of the timed KingJob receives after the last timed step: uint32 counts[pair][5] and fp64 kinship.
    The whole triangle does not fit a comparable dump, so a fixed sample: DUMP_ROWS rows of [r0, r1) and up to
    DUMP_COLS columns of each, drawn by a seeded generator.  Every array is float64 (counts and indices are exact)."""
    import numpy as np

    rng = np.random.default_rng(0)
    lo = max(r0, 1)  # row 0 has no pairs
    rows = np.sort(rng.choice(np.arange(lo, r1), size=min(DUMP_ROWS, r1 - lo), replace=False))
    row_idx, col_idx, counts, kinship = [], [], [], []
    for r in rows:
        r = int(r)
        cols = np.sort(rng.choice(r, size=min(DUMP_COLS, r), replace=False))
        row_idx.append(np.full(cols.size, r))
        col_idx.append(cols)
        counts.append(job.counts(r, r + 1)[cols])  # row r holds the pairs (r, 0..r-1)
        kinship.append(job.kinship(r, r + 1)[cols])
    os.makedirs(out_dir, exist_ok=True)
    for name, parts in (("king_pair_row", row_idx), ("king_pair_col", col_idx), ("king_counts", counts), ("king_kinship", kinship)):
        np.save(os.path.join(out_dir, name + ".npy"), np.concatenate(parts).astype(np.float64))


# ------------------------------------------------------------------------------------- B200 arm
def b200_arm(args):
    import torch
    import torch.distributed as dist

    import plink_ng_b200 as p
    from plink_ng_b200.host import KING_ALGO_POPCOUNT, KING_ALGO_TENSOR, KING_ALGO_TENSOR_TS, KingJob, comm_unique_id
    from plink_ng_b200.sharding import pairs_in_rows, row_block, row_block_tiles, variant_slice

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.samples
    mb = args.batch_variants
    row_bytes = (n + 31) // 32 * 8
    algo = {"tensor_ts": KING_ALGO_TENSOR_TS, "tensor": KING_ALGO_TENSOR, "popcount": KING_ALGO_POPCOUNT}[args.algo]
    if world > 1 and algo != KING_ALGO_TENSOR_TS:
        raise SystemExit("multi-GPU runs use the default (tensor_ts) algorithm")
    r0, r1 = (row_block_tiles if args.row_split == "tiles" else row_block)(n, rank, world)
    my_pairs = pairs_in_rows(r0, r1)
    total_pairs = n * (n - 1) // 2

    # this rank's 1/G slice of the step's variants (rows beyond the slice are all-missing and count nothing)
    per, v0, v1 = variant_slice(mb, rank, world)
    slice_dev = torch.full((per, row_bytes), 0xFF, dtype=torch.uint8, device=dev)
    if v1 > v0:
        slice_dev[: v1 - v0] = synth_genovecs(torch, n, v0, v1, dev)
    torch.cuda.synchronize()

    ctx = p.GpuContext(local_rank)
    if world > 1:
        # NCCL lives in the library: rank 0 creates the id, torch.distributed only ships the 128 bytes
        # (NCCL prints its version banner on stdout at the first communicator init: keep stdout for the one JSON line)
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            ids = [comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            ctx.comm_init(rank, world, ids[0])
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    job = KingJob(ctx, n, r0, r1, algo, max_variants_per_add=per * world)
    ctx.synchronize()

    def step_resident():
        if world == 1:
            job.add_variants_device(slice_dev.data_ptr(), row_bytes, mb, complete=True)
        else:
            job.add_variants_sharded(slice_dev.data_ptr(), row_bytes, per, 2)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launch_count()
    t0 = time.perf_counter()
    ctx.event_record(0)
    for _ in range(args.steps):
        step_resident()
    ctx.event_record(1)
    dev_ms = ctx.event_elapsed_ms(0, 1)
    kern_ms = job.last_kernel_ms() if algo == KING_ALGO_TENSOR_TS else dev_ms / args.steps
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop()
    t_ms = torch.tensor([dev_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    step_ms = float(t_ms[0].item()) / args.steps
    kern_ms_max = float(t_ms[1].item())
    value = total_pairs * (mb / 1e6) / (step_ms * 1e-3)
    # before the e2e leg, which adds more variants to the same job; multi-GPU runs dump rank 0's row block
    if args.dump_outputs and rank == 0:
        dump_outputs(job, r0, r1, args.dump_outputs)

    # ---- e2e: host buffers through the C-ABI, H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        host_slice = torch.empty((per, row_bytes), dtype=torch.uint8, pin_memory=True)
        host_slice.copy_(slice_dev)
        steps_per_job = max(1, -(-FULL_M // mb))
        rows = r1 - r0
        slices = [(r0 + rows * k // steps_per_job, r0 + rows * (k + 1) // steps_per_job) for k in range(steps_per_job)]
        max_pairs = max((b * (b - 1) - a * (a - 1)) // 2 for a, b in slices)
        host_out = torch.empty((max_pairs,), dtype=torch.float64, pin_memory=True)
        import ctypes as C

        from plink_ng_b200.capi import check, lib

        def step_e2e(k):
            if world == 1:
                check(lib.pl2gpu_king_add_variants(job._h, C.c_void_p(host_slice.data_ptr()), row_bytes, mb, 0), "add_variants(host)")
            else:
                check(lib.pl2gpu_king_add_variants_sharded(job._h, C.c_void_p(host_slice.data_ptr()), row_bytes, per, 0), "add_variants_sharded(host)")
            a, b = slices[k % steps_per_job]
            check(lib.pl2gpu_king_get_kinship(job._h, a, b, C.c_void_p(host_out.data_ptr()), 0), "get_kinship(host)")
            return (b * (b - 1) - a * (a - 1)) // 2 * 8

        step_e2e(0)
        barrier()
        t1 = time.perf_counter()
        d2h = 0
        for k in range(args.steps):
            d2h += step_e2e(k)
        barrier()
        e_ms = torch.tensor([(time.perf_counter() - t1) * 1e3], dtype=torch.float64, device=dev)
        d2h_t = torch.tensor([float(d2h)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(d2h_t, op=dist.ReduceOp.SUM)
        e_step_ms = float(e_ms.item()) / args.steps
        e2e = {
            "value": total_pairs * (mb / 1e6) / (e_step_ms * 1e-3), "unit": UNIT,
            "h2d_bytes_per_step": int(per) * int(row_bytes) * world, "d2h_bytes_per_step": int(d2h_t.item() / args.steps),
            "ms_per_step": e_step_ms, "note": "each rank uploads its 1/G slice from pinned host memory; the library all-gathers it over NVLink" if world > 1 else "pinned host batch -> pl2gpu_king_add_variants -> pl2gpu_king_get_kinship into pinned host memory",
        }
        del host_slice, host_out

    job.close()
    if world > 1:
        # tear the library's communicator down on every rank at the same point (ncclCommDestroy synchronises with
        # its peers: closing it on rank 0 while the others already sit in the final torch barrier deadlocks)
        barrier()
        ctx.comm_destroy()
        dist.barrier()
    if rank != 0:
        ctx.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- measured int8 tensor peak of THIS GPU, same run (>= 2 s on all SMs, clocks sampled) ----
    peak, peak_src, peak_detail = 4500.0, "nominal dense int8 4.5 POP/s (measurement failed)", None
    try:
        del slice_dev
        torch.cuda.empty_cache()
        s2 = ClockSampler(local_rank)
        s2.start()
        ts160, secs = ctx.int8_peak(160, 1, 2.0)
        ss240, _ = ctx.int8_peak(240, 0, 0.5)
        pk = s2.stop()
        peak = max(ts160, ss240)
        peak_detail = {"ts_n160_tops": ts160, "ss_n240_tops": ss240, "seconds": secs, "clocks": pk}
        peak_src = "measured in this run: pl2gpu_int8_peak (tcgen05.mma kind::i8, M=128 K=32, all SMs, >= 2 s; max of the A-in-TMEM N=160 form the kernel uses and the smem-smem N=240 form)"
    except Exception as ex:
        peak_src += f": {ex}"
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    ops = 5 * 2 * my_pairs * mb  # algorithmic: 5 indicator products per pair and variant, this rank's launch
    achieved = ops / (kern_ms * 1e-3) / 1e12
    kname = {KING_ALGO_TENSOR_TS: "king_ts_kernel", KING_ALGO_TENSOR: "king_tc_kernel", KING_ALGO_POPCOUNT: "king_popc_kernel"}[algo]
    acc_bytes = 2 * 20 * my_pairs  # int32 x 5 accumulators read + written once per launch (tile padding excluded)
    # DRAM bytes of ONE king_ts_kernel launch at exactly this shape, from `ncu --metrics dram__bytes_read.sum,
    # dram__bytes_write.sum -k regex:king_ts_kernel` on this command (profiles/r02_king_traffic_100k.csv): 609.5 GB read +
    # 100.6 GB written.  Only quoted for the configuration it was captured on.
    traffic = 609530605824 + 100556782336 if (n, mb, world, algo) == (FULL_N, 131072, 1, KING_ALGO_TENSOR_TS) else None
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TOP/s (int8)", "frac": achieved / peak, "traffic": traffic,
                "kernel": kname, "kernel_ms": kern_ms, "kernel_ms_max_over_ranks": kern_ms_max, "peak_source": peak_src, "peak_detail": peak_detail,
                "frac_of_nominal_4500": achieved / 4500.0, "frac_of_2x_bf16_burst": achieved / (2 * peaks["bf16_tflops"]) if peaks.get("bf16_tflops") else None,
                "algorithmic_ops_per_launch": ops, "algorithmic_bytes_per_launch": acc_bytes + n * mb // 2,
                "traffic_note": "bytes per launch from one ncu capture of this kernel at this shape (profiles/r02_king_traffic_100k.csv; profiles/r02_ncu_summary.md has the --set full capture at 16,384 samples): written = the accumulators once (100.6 GB); read = accumulators once + operand tiles re-fetched when the 12x12-tile launch blocks outrun the L2 (15 % of the operand requests miss at 131,072 variants per step). 710 GB in 1.75 s is 6 % of the HBM bandwidth: the kernel is tensor-bound (pipe 82.6 % active) and the re-reads cost no time",
                "kernel_ms_note": "CUDA events recorded by the library around the king_ts_kernel launch on its stream (last timed step); the step additionally holds the copy/all-gather, padding and row re-tiling of the next batch, overlapped on the prep stream"}
    if algo == KING_ALGO_POPCOUNT:
        roofline["note"] = "popcount kernel: int8-equivalent ops shown for comparability; its own limiter is the POPC pipe"

    secondary = None
    if world == 1 and not args.no_secondary:
        secondary = secondary_legs(args, torch, p, ctx, dev, peak)
    ctx.close()
    cpu_baseline, cli = (None, None)
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, cli = cpu_legs(args)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32 popcount" if algo == KING_ALGO_POPCOUNT else "s8 (exact int32 accumulate)",
        "data": "synthetic",
        "config": {"workload": f"--make-king, {n} samples x {FULL_M} SNPs in steps of {mb} variants", "samples": n, "variants_per_step": mb, "steps_per_full_job": -(-FULL_M // mb),
                   "parallelism": f"row-block x{world} ({'tile-aligned equal work' if args.row_split == 'tiles' else 'ParallelBounds'}), 1 NCCL all-gather of the genotype column tile per step inside libpl2gpu, overlapped" if world > 1 else "single GPU",
                   "algo": args.algo, "rows_rank0": [r0, r1],
                   "l2_policy": "inputs (3.3 GB batch + 100 GB of accumulators) exceed L2; no flush needed", "pair_snp_per_s": total_pairs * mb / (step_ms * 1e-3), "wall_ms_per_step": wall_ms / args.steps},
        "roofline": roofline, "cpu_baseline": cpu_baseline, "cli_same_files": cli, "secondary": secondary, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
    }
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_JSON_FD = None


def emit(line):
    """The ONE JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    args = parse_args()
    # Libraries print banners on stdout (NCCL's "NCCL version ..." at the first communicator init, from torch's
    # bundled copy as well as from the one libpl2gpu loads): everything but the JSON line goes to stderr.
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
