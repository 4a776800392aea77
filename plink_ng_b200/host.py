"""Thin host-side mirror of the reference's calling conventions for tests and bench.py.

Names follow the reference: `parallel_bounds` is ParallelBounds (2.0/plink2_common.cc:4956),
genotype blocks are "genovecs" in PgrGet layout (2.0/include/pgenlib_read.h:537), KING results are
`king_counts[pair][5]` (2.0/plink2_matrix_calc.cc:864-868).
"""
import ctypes as C
import math

import numpy as np

from . import capi
from .capi import lib, check

KING_ALGO_AUTO, KING_ALGO_POPCOUNT, KING_ALGO_TENSOR, KING_ALGO_TENSOR_TS = 0, 1, 2, 3


def pack_genotypes(geno: np.ndarray) -> np.ndarray:
    """[variants, samples] uint8 codes (0,1,2 = ALT dosage, 3 = missing) -> genovecs
    [variants, ceil(samples/32)] uint64 in PgrGet layout (trailing entries zero)."""
    geno = np.ascontiguousarray(geno, dtype=np.uint8)
    m, n = geno.shape
    n32 = (n + 31) // 32 * 32
    pad = np.zeros((m, n32), dtype=np.uint8)
    pad[:, :n] = geno & 3
    q = pad.reshape(m, n32 // 4, 4)
    by = (q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)).astype(np.uint8)
    return np.ascontiguousarray(by).view("<u8").reshape(m, n32 // 32)


def unpack_genotypes(genovecs: np.ndarray, sample_ct: int) -> np.ndarray:
    by = np.ascontiguousarray(genovecs).view(np.uint8).reshape(genovecs.shape[0], -1)
    codes = np.stack([(by >> s) & 3 for s in (0, 2, 4, 6)], axis=-1).reshape(by.shape[0], -1)
    return np.ascontiguousarray(codes[:, :sample_ct])


def _triangle_divide(cur_prod_x2: int, modif: int) -> int:
    # 2.0/plink2_common.cc:4936-4954
    if cur_prod_x2 == 0:
        return -modif if modif < 0 else 0
    vv = int(math.sqrt(float(cur_prod_x2)))
    while (vv - 1) * (vv + modif - 1) >= cur_prod_x2:
        vv -= 1
    while vv * (vv + modif) < cur_prod_x2:
        vv += 1
    return vv


def parallel_bounds(ct: int, start: int, parallel_idx: int, parallel_tot: int):
    """ParallelBounds (2.0/plink2_common.cc:4956-4961): equal-area row range of piece k of n."""
    modif = 1 - start * 2
    ct_tot = ct * (ct + modif)
    return (
        _triangle_divide((ct_tot * parallel_idx) // parallel_tot, modif),
        _triangle_divide((ct_tot * (parallel_idx + 1)) // parallel_tot, modif),
    )


class GpuContext:
    def __init__(self, device_idx: int = 0):
        self._h = C.c_void_p()
        check(lib.pl2gpu_ctx_create(device_idx, C.byref(self._h)), "pl2gpu_ctx_create")

    @property
    def handle(self):
        return self._h

    def synchronize(self):
        check(lib.pl2gpu_ctx_synchronize(self._h), "pl2gpu_ctx_synchronize")

    def launch_count(self) -> int:
        return int(lib.pl2gpu_ctx_launch_count(self._h))

    def event_record(self, slot: int):
        check(lib.pl2gpu_ctx_event_record(self._h, slot), "pl2gpu_ctx_event_record")

    def event_elapsed_ms(self, slot_from: int, slot_to: int) -> float:
        ms = C.c_float()
        check(lib.pl2gpu_ctx_event_elapsed_ms(self._h, slot_from, slot_to, C.byref(ms)), "pl2gpu_ctx_event_elapsed_ms")
        return float(ms.value)

    def stream(self) -> int:
        return int(lib.pl2gpu_ctx_stream(self._h) or 0)

    def int8_peak(self, n_cols: int = 160, form: int = 1, min_seconds: float = 2.0):
        """Measured chip-wide tcgen05 kind::i8 rate (TOP/s, seconds): the roofline denominator."""
        tops, secs = C.c_double(), C.c_double()
        check(lib.pl2gpu_int8_peak(self._h, n_cols, form, min_seconds, C.byref(tops), C.byref(secs)), "pl2gpu_int8_peak")
        return float(tops.value), float(secs.value)

    def mxf4_peak(self, n_cols: int = 160, min_seconds: float = 2.0):
        """Measured chip-wide tcgen05 kind::mxf4 rate (TOP/s, seconds), A operand in tensor memory."""
        tops, secs = C.c_double(), C.c_double()
        check(lib.pl2gpu_mxf4_peak(self._h, n_cols, min_seconds, C.byref(tops), C.byref(secs)), "pl2gpu_mxf4_peak")
        return float(tops.value), float(secs.value)

    def comm_init(self, rank: int, world: int, unique_id: bytes):
        """Attach an NCCL communicator (collective over all ranks; rank 0 makes the id with comm_unique_id())."""
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        check(lib.pl2gpu_comm_init(self._h, rank, world, buf), "pl2gpu_comm_init")

    def comm_destroy(self):
        """Collective teardown of the communicator (every rank calls it at the same point); idempotent."""
        check(lib.pl2gpu_comm_destroy(self._h), "pl2gpu_comm_destroy")

    def selftest_umma(self, verbose: bool = True):
        check(lib.pl2gpu_selftest_umma(self._h, 1 if verbose else 0), "pl2gpu_selftest_umma")

    def close(self):
        if self._h:
            lib.pl2gpu_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def comm_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    check(lib.pl2gpu_comm_unique_id(buf), "pl2gpu_comm_unique_id")
    return bytes(buf)


def _pairs(r0: int, r1: int) -> int:
    tri = lambda r: r * (r - 1) // 2 if r else 0  # noqa: E731
    return tri(r1) - tri(r0)


class KingJob:
    """CalcKing's dense loop (2.0/plink2_matrix_calc.cc:2016-2117) for one row range."""

    def __init__(self, ctx: GpuContext, sample_ct: int, row_start: int = 0, row_end: int = None, algo: int = KING_ALGO_AUTO, max_variants_per_add: int = 0):
        self.ctx = ctx
        self.sample_ct = sample_ct
        self.row_start = row_start
        self.row_end = sample_ct if row_end is None else row_end
        self._h = C.c_void_p()
        check(lib.pl2gpu_king_begin_ex(ctx.handle, sample_ct, self.row_start, self.row_end, algo, max_variants_per_add, C.byref(self._h)), "pl2gpu_king_begin_ex")

    def add_variants(self, genovecs: np.ndarray):
        """genovecs: host uint64 [variants, ceil(sample_ct/32)] (PgrGet rows)."""
        g = np.ascontiguousarray(genovecs)
        assert g.dtype == np.uint64 and g.ndim == 2 and g.shape[1] * 32 >= self.sample_ct
        check(lib.pl2gpu_king_add_variants(self._h, g.ctypes.data, g.strides[0], g.shape[0], 0), "pl2gpu_king_add_variants")

    def add_variants_device(self, dev_ptr: int, stride_bytes: int, variant_ct: int, complete: bool = False):
        """complete=True: the device buffer is not being written by pending work (src_is_device = 2)."""
        check(lib.pl2gpu_king_add_variants(self._h, C.c_void_p(dev_ptr), stride_bytes, variant_ct, 2 if complete else 1), "pl2gpu_king_add_variants")

    def add_variants_sharded(self, ptr: int, stride_bytes: int, slice_variant_ct: int, src_is_device: int):
        """Collective: this rank's slice of the batch; the library all-gathers the column tile (NCCL)."""
        check(lib.pl2gpu_king_add_variants_sharded(self._h, C.c_void_p(ptr), stride_bytes, slice_variant_ct, src_is_device), "pl2gpu_king_add_variants_sharded")

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        check(lib.pl2gpu_king_last_kernel_ms(self._h, C.byref(ms)), "pl2gpu_king_last_kernel_ms")
        return float(ms.value)

    def counts(self, row_start: int = None, row_end: int = None) -> np.ndarray:
        r0 = self.row_start if row_start is None else row_start
        r1 = self.row_end if row_end is None else row_end
        out = np.empty((_pairs(r0, r1), 5), dtype=np.uint32)
        check(lib.pl2gpu_king_get_counts(self._h, r0, r1, out.ctypes.data, 0), "pl2gpu_king_get_counts")
        return out

    def kinship(self, row_start: int = None, row_end: int = None) -> np.ndarray:
        r0 = self.row_start if row_start is None else row_start
        r1 = self.row_end if row_end is None else row_end
        out = np.empty(_pairs(r0, r1), dtype=np.float64)
        check(lib.pl2gpu_king_get_kinship(self._h, r0, r1, out.ctypes.data, 0), "pl2gpu_king_get_kinship")
        return out

    def filtered(self, min_kinship: float, max_out: int = 1 << 20, row_start: int = None, row_end: int = None):
        """--king-table-filter on the device: (pairs [k,2] = (j, i), counts [k,5], kinship [k]) in table order,
        only pairs whose kinship is not below min_kinship.  Grows the buffers and retries on overflow."""
        r0 = self.row_start if row_start is None else row_start
        r1 = self.row_end if row_end is None else row_end
        while True:
            pairs = np.empty((max_out, 2), dtype=np.uint32)
            counts = np.empty((max_out, 5), dtype=np.uint32)
            kin = np.empty(max_out, dtype=np.float64)
            found = C.c_uint64(0)
            check(lib.pl2gpu_king_get_filtered(self._h, r0, r1, min_kinship, max_out, pairs.ctypes.data, counts.ctypes.data, kin.ctypes.data, C.byref(found)), "pl2gpu_king_get_filtered")
            if found.value <= max_out:
                k = found.value
                return pairs[:k], counts[:k], kin[:k]
            max_out = int(found.value)

    def counts_to_device(self, dev_ptr: int, row_start: int, row_end: int):
        check(lib.pl2gpu_king_get_counts(self._h, row_start, row_end, C.c_void_p(dev_ptr), 1), "pl2gpu_king_get_counts")

    def kinship_to_device(self, dev_ptr: int, row_start: int, row_end: int):
        check(lib.pl2gpu_king_get_kinship(self._h, row_start, row_end, C.c_void_p(dev_ptr), 1), "pl2gpu_king_get_kinship")

    def close(self):
        if self._h:
            lib.pl2gpu_king_end(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class KingPairJob:
    """KING counts for an explicit pair list (`--king-table-subset`; CalcKingTableSubset,
    2.0/plink2_matrix_calc.cc:3224).  pairs: int array [P, 2] of sample indices (first, second)."""

    def __init__(self, ctx: GpuContext, sample_ct: int, pairs: np.ndarray):
        self.pairs = np.ascontiguousarray(pairs, dtype=np.uint32).reshape(-1, 2)
        self.sample_ct = sample_ct
        self._h = C.c_void_p()
        check(lib.pl2gpu_king_pairs_begin(ctx.handle, sample_ct, self.pairs.ctypes.data, len(self.pairs), C.byref(self._h)), "pl2gpu_king_pairs_begin")

    def add_variants(self, genovecs: np.ndarray):
        g = np.ascontiguousarray(genovecs)
        check(lib.pl2gpu_king_pairs_add_variants(self._h, g.ctypes.data, g.strides[0], g.shape[0], 0), "pl2gpu_king_pairs_add_variants")

    def counts(self) -> np.ndarray:
        out = np.empty((len(self.pairs), 5), dtype=np.uint32)
        check(lib.pl2gpu_king_pairs_get_counts(self._h, 0, len(self.pairs), out.ctypes.data, 0), "pl2gpu_king_pairs_get_counts")
        return out

    def close(self):
        if self._h:
            lib.pl2gpu_king_pairs_end(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def king_counts(genovecs: np.ndarray, sample_ct: int, algo: int = KING_ALGO_AUTO, device: int = 0, batch: int = 65536) -> np.ndarray:
    """All-pairs king_counts[pair][5] for one genotype block (convenience for tests)."""
    with GpuContext(device) as ctx, KingJob(ctx, sample_ct, 0, sample_ct, algo) as job:
        for s in range(0, genovecs.shape[0], batch):
            job.add_variants(genovecs[s : s + batch])
        return job.counts()


def geno_counts(ctx: GpuContext, genovecs: np.ndarray, sample_ct: int) -> np.ndarray:
    """uint32 [variants, 4] = {hom-REF, het, hom-ALT, missing} (GenoarrCountFreqsUnsafe)."""
    g = np.ascontiguousarray(genovecs)
    out = np.empty((g.shape[0], 4), dtype=np.uint32)
    check(lib.pl2gpu_geno_counts(ctx.handle, g.ctypes.data, g.strides[0], sample_ct, g.shape[0], 0, out.ctypes.data), "pl2gpu_geno_counts")
    return out


def ld_band_flags(ctx: GpuContext, genovecs: np.ndarray, founder_ct: int, band: int, prune_ld_thresh: float) -> np.ndarray:
    g = np.ascontiguousarray(genovecs)
    out = np.zeros((g.shape[0], band), dtype=np.uint8)
    check(lib.pl2gpu_ld_band_flags(ctx.handle, g.ctypes.data, g.strides[0], founder_ct, g.shape[0], 0, band, prune_ld_thresh, out.ctypes.data), "pl2gpu_ld_band_flags")
    return out


def indep_pairwise(ctx: GpuContext, genovecs: np.ndarray, founder_ct: int, chr_codes, bps, window: int, step: int, r2: float, window_is_bp: bool = False, ref_freqs=None, preferred=None) -> np.ndarray:
    """LdPrune/IndepPairwise (2.0/plink2_ld.cc:2530) on an in-memory block -> removed[variants] uint8."""
    g = np.ascontiguousarray(genovecs)
    m = g.shape[0]
    chr_codes = np.ascontiguousarray(chr_codes, dtype=np.uint32)
    bps_a = np.ascontiguousarray(bps, dtype=np.uint32) if bps is not None else None
    rf = np.ascontiguousarray(ref_freqs, dtype=np.float64) if ref_freqs is not None else None
    pf = np.ascontiguousarray(preferred, dtype=np.uint8) if preferred is not None else None
    out = np.zeros(m, dtype=np.uint8)
    check(
        lib.pl2_indep_pairwise(ctx.handle, g.ctypes.data, g.strides[0], founder_ct, m, chr_codes.ctypes.data, bps_a.ctypes.data if bps_a is not None else None,
                               window, step, r2, 1 if window_is_bp else 0, rf.ctypes.data if rf is not None else None, pf.ctypes.data if pf is not None else None, 0, out.ctypes.data),
        "pl2_indep_pairwise",
    )
    return out


GRM_MEANIMPUTE, GRM_COV = 1, 2


class GrmJob:
    """CalcGrm's accumulation loop (2.0/plink2_matrix_calc.cc:4711-4749) for one row range."""

    def __init__(self, ctx: GpuContext, sample_ct: int, row_start: int = 0, row_end: int = None, flags: int = 0):
        self.ctx = ctx
        self.sample_ct = sample_ct
        self.row_start = row_start
        self.row_end = sample_ct if row_end is None else row_end
        self._h = C.c_void_p()
        check(lib.pl2gpu_grm_begin(ctx.handle, sample_ct, self.row_start, self.row_end, flags, C.byref(self._h)), "pl2gpu_grm_begin")

    def add_variants(self, genovecs: np.ndarray, ref_freqs=None):
        g = np.ascontiguousarray(genovecs)
        rf = None if ref_freqs is None else np.ascontiguousarray(ref_freqs, dtype=np.float64)
        rc = lib.pl2gpu_grm_add_variants(self._h, g.ctypes.data, g.strides[0], g.shape[0], 0, rf.ctypes.data if rf is not None else None)
        check(rc, "pl2gpu_grm_add_variants")

    def add_variants_device(self, dev_ptr: int, stride_bytes: int, variant_ct: int, ref_freqs=None):
        rf = None if ref_freqs is None else np.ascontiguousarray(ref_freqs, dtype=np.float64)
        check(lib.pl2gpu_grm_add_variants(self._h, C.c_void_p(dev_ptr), stride_bytes, variant_ct, 1, rf.ctypes.data if rf is not None else None), "pl2gpu_grm_add_variants")

    def rows(self, r0: int = None, r1: int = None, with_obs: bool = False):
        r0 = self.row_start if r0 is None else r0
        r1 = self.row_end if r1 is None else r1
        g = np.zeros((r1 - r0, r1), dtype=np.float64)
        obs = np.zeros((r1 - r0, r1), dtype=np.float32) if with_obs else None
        check(lib.pl2gpu_grm_get_rows(self._h, r0, r1, g.ctypes.data, obs.ctypes.data if with_obs else None, r1, 0), "pl2gpu_grm_get_rows")
        return (g, obs) if with_obs else g

    def eigen_topk(self, pc_ct: int):
        """Exact --pca: (eigvals[pc_ct] descending, eigvecs[pc_ct, samples])."""
        vals = np.empty(pc_ct, dtype=np.float64)
        vecs = np.empty((pc_ct, self.sample_ct), dtype=np.float64)
        check(lib.pl2gpu_grm_eigen_topk(self._h, pc_ct, vals.ctypes.data, vecs.ctypes.data), "pl2gpu_grm_eigen_topk")
        return vals, vecs

    def close(self):
        if self._h:
            lib.pl2gpu_grm_end(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def pca_approx(ctx: GpuContext, genovecs: np.ndarray, sample_ct: int, pc_ct: int, g1: np.ndarray, ref_freqs=None):
    """`--pca approx` on an in-memory block with a caller-supplied Gaussian start matrix
    g1 [sample_ct, 2*pc_ct] -> (eigvals[pc_ct], eigvecs[pc_ct, sample_ct])."""
    g = np.ascontiguousarray(genovecs)
    g1 = np.ascontiguousarray(g1, dtype=np.float64)
    assert g1.shape == (sample_ct, 2 * pc_ct)
    rf = None if ref_freqs is None else np.ascontiguousarray(ref_freqs, dtype=np.float64)
    h = C.c_void_p()
    check(lib.pl2gpu_pca_begin(ctx.handle, sample_ct, g.shape[0], pc_ct, C.byref(h)), "pl2gpu_pca_begin")
    try:
        check(lib.pl2gpu_pca_add_variants(h, g.ctypes.data, g.strides[0], g.shape[0], 0, rf.ctypes.data if rf is not None else None), "pl2gpu_pca_add_variants")
        vals = np.empty(pc_ct, dtype=np.float64)
        vecs = np.empty((pc_ct, sample_ct), dtype=np.float64)
        check(lib.pl2gpu_pca_run(h, g1.ctypes.data, vals.ctypes.data, vecs.ctypes.data), "pl2gpu_pca_run")
        return vals, vecs
    finally:
        lib.pl2gpu_pca_end(h)


def score_sums(ctx: GpuContext, genovecs: np.ndarray, sample_ct: int, weights4: np.ndarray, named_dosages: np.ndarray):
    """`--score` accumulation (pl2gpu_score_*) over an in-memory block of scored entries: genovecs [entries, words]
    PgrGet rows, weights4 [entries, 4] fp64 contributions of genotype codes 0..3, named_dosages [entries] uint8
    (dosages of codes 0, 1, 2 packed two bits each) -> (score sums, named-allele dosage sums, missing counts)."""
    g = np.ascontiguousarray(genovecs)
    w = np.ascontiguousarray(weights4, dtype=np.float64)
    d = np.ascontiguousarray(named_dosages, dtype=np.uint8)
    assert w.shape == (g.shape[0], 4) and d.shape == (g.shape[0],)
    h = C.c_void_p()
    check(lib.pl2gpu_score_begin(ctx.handle, sample_ct, C.byref(h)), "pl2gpu_score_begin")
    try:
        check(lib.pl2gpu_score_add_variants(h, g.ctypes.data, g.strides[0], g.shape[0], 0, w.ctypes.data, d.ctypes.data), "pl2gpu_score_add_variants")
        sums = np.empty(sample_ct, dtype=np.float64)
        dos = np.empty(sample_ct, dtype=np.uint64)
        miss = np.empty(sample_ct, dtype=np.uint32)
        check(lib.pl2gpu_score_get(h, sums.ctypes.data, dos.ctypes.data, miss.ctypes.data), "pl2gpu_score_get")
        return sums, dos, miss
    finally:
        lib.pl2gpu_score_end(h)


def variant_scores(ctx: GpuContext, genovecs: np.ndarray, sample_ct: int, weights: np.ndarray, ref_freqs=None) -> np.ndarray:
    """`--variant-score` sums (pl2gpu_pca_vscore) for an in-memory block: weights [sample_ct, cols] -> [variants, cols]."""
    g = np.ascontiguousarray(genovecs)
    w = np.ascontiguousarray(weights, dtype=np.float64)
    assert w.shape[0] == sample_ct
    rf = None if ref_freqs is None else np.ascontiguousarray(ref_freqs, dtype=np.float64)
    h = C.c_void_p()
    check(lib.pl2gpu_pca_begin_shard(ctx.handle, sample_ct, g.shape[0], 1, C.byref(h)), "pl2gpu_pca_begin_shard")
    try:
        check(lib.pl2gpu_pca_add_variants(h, g.ctypes.data, g.strides[0], g.shape[0], 0, rf.ctypes.data if rf is not None else None), "pl2gpu_pca_add_variants")
        out = np.empty((g.shape[0], w.shape[1]), dtype=np.float64)
        check(lib.pl2gpu_pca_vscore(h, w.ctypes.data, w.shape[1], out.ctypes.data), "pl2gpu_pca_vscore")
        return out
    finally:
        lib.pl2gpu_pca_end(h)
