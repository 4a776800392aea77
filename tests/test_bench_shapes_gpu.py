"""KING at the shapes and through the entry points bench.py uses, checked exactly against an independent reference.

`king_ref_counts` evaluates the five KING sums for a sample of pairs as indicator-matrix products in float64 (exact
below 2^53), with numpy on the host or torch (cuBLAS) on the device, never through libpl2gpu.  The non-GPU test
pins it to the oracle's per-pair restatements.

The GPU tests cover what the rest of the suite does not reach:
  - the benchmark's job: 100,000 samples (490,156 TS tiles, 2.5e10 accumulator words, so tile and pair offsets
    pass 2^32), 131,072-variant launches fed by add_variants_device(complete=True), relatives planted at known
    places, read back through counts / kinship / filtered / counts_to_device / kinship_to_device;
  - many waves with a small stage cap, so one call splits into several launches over both TS stage buffers, device
    sources rewritten on the context's stream right after the call, a source written on that stream just before
    a complete=False call, and a row block that is not tile-aligned, against the popcount kernel."""
import ctypes as C

import numpy as np
import pytest

from oracle import plink_oracle as orc
from plink_ng_b200.capi import check, lib
from plink_ng_b200.host import KING_ALGO_POPCOUNT, KING_ALGO_TENSOR_TS, KingJob

KING_NAMES = ("IBS0", "HETHET", "HET2HOM1", "HET1HOM2", "HOMHOM")


def king_ref_counts(codes_r, codes_c, chunk=8192):
    """The five KING count matrices {IBS0, HETHET, HET2HOM1, HET1HOM2, HOMHOM} of row samples R against column
    samples C, as int64 numpy [5, |R|, |C|], from 2-bit codes [variants, |R|] and [variants, |C|] (0 hom-REF,
    1 het, 2 hom-ALT, 3 missing).  Orientation of oracle.king_count_matrices: the row sample is the pair's second
    (larger-index) sample, so HET2HOM1[r, c] = het_r . hom_c.  numpy arrays are evaluated on the host, torch
    tensors on their device; either way as float64 products of 0/1 indicators, exact below 2^53."""
    if isinstance(codes_r, np.ndarray):
        xp, f64 = np, (lambda x: x.astype(np.float64))
    else:
        import torch

        xp, f64 = torch, (lambda x: x.to(torch.float64))
    acc = None
    for v0 in range(0, codes_r.shape[0], chunk):
        a, b = codes_r[v0 : v0 + chunk], codes_c[v0 : v0 + chunk]
        ra, ha, aa = f64(a == 0), f64(a == 1), f64(a == 2)
        rb, hb, ab = f64(b == 0), f64(b == 1), f64(b == 2)
        oa, ob = ra + aa, rb + ab  # homozygous
        part = xp.stack([ra.T @ ab + aa.T @ rb, ha.T @ hb, ha.T @ ob, oa.T @ hb, oa.T @ ob])
        acc = part if acc is None else acc + part
    if acc is None:
        return np.zeros((5, codes_r.shape[1], codes_c.shape[1]), dtype=np.int64)
    acc = acc if xp is np else acc.cpu().numpy()
    return np.rint(acc).astype(np.int64)


def _random_codes(m, n, seed, miss=0.05):
    rng = np.random.default_rng(seed)
    freq = rng.uniform(0.02, 0.98, size=(m, 1))
    g = (rng.random((m, n)) < freq).astype(np.uint8) + (rng.random((m, n)) < freq).astype(np.uint8)
    g[rng.random((m, n)) < miss] = 3
    return g


@pytest.mark.parametrize("n,m,seed", [(2, 1, 0), (9, 40, 1), (37, 300, 2), (61, 9000, 3)])
def test_king_ref_counts_matches_oracle(n, m, seed):
    """The reference against oracle.king_counts_pairs (the explicit per-pair restatement) and, on the small inputs,
    oracle.king_counts_bruteforce (the literal per-genotype table), with row and column sets in both orders and
    chunk boundaries inside the variants."""
    geno = _random_codes(m, n, seed)
    geno[:, n - 1] = 3  # an all-missing sample
    rng = np.random.default_rng(seed + 100)
    rows = rng.choice(n, size=min(n, 7), replace=False)
    cols = rng.choice(n, size=min(n, 11), replace=False)
    got = king_ref_counts(geno[:, rows], geno[:, cols], chunk=97)
    assert got.shape == (5, len(rows), len(cols))
    pairs = np.array([(c, r) for r in rows for c in cols], dtype=np.int64)  # (first, second): "2" is the row sample
    want = orc.king_counts_pairs(geno, pairs).astype(np.int64).reshape(len(rows), len(cols), 5)
    assert np.array_equal(got, want.transpose(2, 0, 1))
    if n * n * m <= 1_000_000:
        brute = orc.king_counts_bruteforce(geno).astype(np.int64)  # pair (i, j), i < j, at j (j - 1) / 2 + i
        for ri, r in enumerate(rows):
            for ci, c in enumerate(cols):
                if c < r:
                    assert np.array_equal(got[:, ri, ci], brute[r * (r - 1) // 2 + c]), (r, c)
    np.testing.assert_array_equal(king_ref_counts(geno[:0, rows], geno[:0, cols]), 0)


# ------------------------------------------------------------------------------------------------ device helpers
def _sample_codes(g, samples):
    """Codes [variants, len(samples)] (uint8, same device) of the given samples of a device genovec tensor
    g = uint8 [variants, row_bytes] in PgrGet layout: sample s sits in byte s // 4 at bit 2 * (s % 4)."""
    import torch

    idx = torch.as_tensor(np.asarray(samples, dtype=np.int64), device=g.device)
    return (g[:, idx // 4] >> (2 * (idx % 4)).to(torch.uint8)) & 3


def _set_codes(g, s, codes):
    """Overwrite sample s's codes (uint8 [variants] on g's device) in the genovec tensor g."""
    sh = 2 * (s % 4)
    col = g[:, s // 4]
    g[:, s // 4] = (col & (0xFF ^ (3 << sh))) | (codes << sh)


def _pairs_before(r0, r1):
    tri = lambda r: r * (r - 1) // 2 if r else 0  # noqa: E731
    return tri(r1) - tri(r0)


# ------------------------------------------------------------------------------------------ 1. the benchmark's job
N_BENCH = 100_000
STEP = 131_072
STEPS = 3
DUP_OF, DUP_AT = 3, 99_999  # exact duplicate
HALF_OF, HALF_AT = 94_999, 95_000  # half the variants copied: kinship ~0.25
CORNER_COL, CORNER_ROW = 30_000, 60_031  # 30,000 = 375 x 80 opens a column tile, 60,031 = 468 x 128 + 127 closes a row tile
PLANTED = [(CORNER_ROW, CORNER_COL), (HALF_AT, HALF_OF), (DUP_AT, DUP_OF)]  # (j, i) in table order
RANGE_ROWS = (92_600, 92_760)  # the pair index passes 2^32 between rows 92,682 and 92,683


def _bench_sample():
    """Seeded rows R (64) and columns C (about 4,500) of the pair sample; row r is compared at the columns c < r."""
    rng = np.random.default_rng(2026)
    n_rt = -(-N_BENCH // 128)
    last_band_row0 = (n_rt - 1) // 12 * 12 * 128  # first row of BuildTileList's last 12 x 12-tile launch band
    # 41,344-41,471: the row tile holding TS tile 83,886, the first whose accumulator word offset passes 2^32
    fixed = [1, 127, 128, 92_682, 92_683, 99_968, DUP_AT, HALF_AT, CORNER_ROW, 640, 1535, last_band_row0, last_band_row0 + 79, 41_344, 41_471]
    fixed += [int(x) for x in rng.choice(np.arange(2, 12 * 128), size=3, replace=False)]  # first launch band
    fixed += [int(x) for x in rng.choice(np.arange(last_band_row0, N_BENCH), size=3, replace=False)]  # last launch band
    rest = rng.choice(np.setdiff1d(np.arange(2, N_BENCH), fixed), size=64 - len(set(fixed)), replace=False)
    rows = np.unique(np.concatenate([np.array(fixed), rest]))
    cols = set(int(x) for x in rng.choice(N_BENCH - 1, size=4096, replace=False)) | {0, 79, 80, 159, 160, DUP_OF, HALF_OF, CORNER_COL}
    for r in rows:
        m80 = int(r) // 80 * 80
        cols |= {int(r) - 1, m80, m80 - 1, m80 - 80, m80 - 81}
    cols = np.array(sorted(c for c in cols if 0 <= c < N_BENCH), dtype=np.int64)
    assert len(rows) == 64
    return rows.astype(np.int64), cols


def _plant(g, step):
    """Known relatives in one step's genovecs (device, in place)."""
    import torch

    _set_codes(g, DUP_AT, _sample_codes(g, [DUP_OF])[:, 0].contiguous())
    _set_codes(g, CORNER_ROW, _sample_codes(g, [CORNER_COL])[:, 0].contiguous())
    gen = torch.Generator(device=g.device)
    gen.manual_seed(77 + step)
    take = torch.rand(g.shape[0], generator=gen, device=g.device) < 0.5
    both = _sample_codes(g, [HALF_OF, HALF_AT])
    _set_codes(g, HALF_AT, torch.where(take, both[:, 0], both[:, 1]).contiguous())


@pytest.fixture(scope="class")
def bench_job(gpu_ctx):
    """One job as bench.py builds it (all 100,000 rows, TS kernel, 131,072 variants per add, device-resident input),
    three steps of distinct data, and the exact reference on 64 rows x ~4,500 columns accumulated alongside.
    Class-scoped: its 115 GB are released before the other tests of this file run."""
    import torch

    from bench import synth_genovecs

    dev = torch.device("cuda", 0)
    row_bytes = (N_BENCH + 31) // 32 * 8
    need = int(lib.pl2gpu_king_mem_required(N_BENCH, 0, N_BENCH, STEP)) + STEP * row_bytes
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need + (8 << 30):  # + data generation and the reference's working set
        pytest.skip(f"the 100,000-sample job needs {need / 1e9:.1f} GB (+8 GB working set); {free / 1e9:.1f} GB free")
    rows, cols = _bench_sample()
    ref = np.zeros((5, len(rows), len(cols)), dtype=np.int64)
    job = KingJob(gpu_ctx, N_BENCH, 0, N_BENCH, KING_ALGO_TENSOR_TS, max_variants_per_add=STEP)
    try:
        for k in range(STEPS):
            gpu_ctx.synchronize()  # the previous step's copy (queued before its kernel) is done: its buffer may go
            g = synth_genovecs(torch, N_BENCH, k * STEP, (k + 1) * STEP, dev)
            _plant(g, k)
            torch.cuda.synchronize()
            job.add_variants_device(g.data_ptr(), row_bytes, STEP, complete=True)
            ref += king_ref_counts(_sample_codes(g, rows), _sample_codes(g, cols))
            torch.cuda.synchronize()
        gpu_ctx.synchronize()
        del g
        torch.cuda.empty_cache()
        yield job, rows, cols, ref
    finally:
        job.close()


@pytest.mark.gpu
class TestKingBenchShape:
    """Counts, kinship, the table filter and the row-range downloads of the bench_job."""

    def test_sampled_counts_and_kinship_exact(self, bench_job):
        job, rows, cols, ref = bench_job
        assert int(lib.pl2gpu_king_variants_added(job._h)) == STEPS * STEP
        for ri, r in enumerate(rows):
            r = int(r)
            sel = cols < r
            got = job.counts(r, r + 1)[cols[sel]].astype(np.int64)  # row r holds the pairs (r, 0..r-1)
            want = ref[:, ri, sel].T
            for q, name in enumerate(KING_NAMES):
                bad = np.flatnonzero(got[:, q] != want[:, q])
                assert bad.size == 0, f"row {r}: {name} differs at columns {cols[sel][bad[:8]].tolist()} ({bad.size} of {sel.sum()})"
            kin = job.kinship(r, r + 1)[cols[sel]]
            wk = orc.king_kinship(want)
            assert np.array_equal(kin, wk, equal_nan=True), r  # same integers, one IEEE divide: bit for bit

    def test_planted_relatives_and_filter(self, bench_job):
        job, rows, cols, ref = bench_job
        kin_at = {}
        unrelated = []
        planted = set(PLANTED)
        for ri, r in enumerate(rows):
            sel = np.flatnonzero(cols < r)
            wk = orc.king_kinship(ref[:, ri, sel].T)
            for c, k in zip(cols[sel], wk):
                if (int(r), int(c)) in planted:
                    kin_at[(int(r), int(c))] = k
                else:
                    unrelated.append(k)
        unrelated = np.array(unrelated)
        assert set(kin_at) == planted
        assert kin_at[(DUP_AT, DUP_OF)] == 0.5 and kin_at[(CORNER_ROW, CORNER_COL)] == 0.5
        assert 0.2 < kin_at[(HALF_AT, HALF_OF)] < 0.3
        # the 0.1 threshold sits well clear of every unrelated pair in the sample (HWE data, 393,216 variants)
        assert not np.isnan(unrelated).any() and np.abs(unrelated).max() < 0.05, np.abs(unrelated).max()
        found = C.c_uint64(0)  # count first: a broken filter must not make filtered() grow its buffers to 5e9 pairs
        check(lib.pl2gpu_king_get_filtered(job._h, 0, N_BENCH, 0.1, 0, None, None, None, C.byref(found)), "pl2gpu_king_get_filtered")
        assert found.value == len(PLANTED), found.value
        pairs, counts, kin = job.filtered(0.1, 16, 0, N_BENCH)
        assert [tuple(int(x) for x in p) for p in pairs] == PLANTED
        for (j, i), c, k in zip(PLANTED, counts, kin):
            want = ref[:, np.searchsorted(rows, j), np.searchsorted(cols, i)]
            assert np.array_equal(c.astype(np.int64), want), (j, i)
            assert k == orc.king_kinship(want[None])[0]

    def test_row_range_across_2_32_host_and_device(self, bench_job):
        import torch

        job, rows, cols, ref = bench_job
        r0, r1 = RANGE_ROWS
        pairs = _pairs_before(r0, r1)
        assert _pairs_before(0, r0) < (1 << 32) < _pairs_before(0, r1)
        host = job.counts(r0, r1)  # 14.8 M pairs: more than the library's 256 MB download staging
        dev_out = torch.empty(pairs * 5, dtype=torch.int32, device="cuda")
        job.counts_to_device(dev_out.data_ptr(), r0, r1)
        host_kin = job.kinship(r0, r1)
        dev_kin = torch.empty(pairs, dtype=torch.float64, device="cuda")
        job.kinship_to_device(dev_kin.data_ptr(), r0, r1)
        job.ctx.synchronize()
        assert np.array_equal(dev_out.cpu().numpy().view(np.uint32).reshape(pairs, 5), host)
        assert np.array_equal(dev_kin.cpu().numpy(), host_kin, equal_nan=True)
        checked = 0
        for ri, r in enumerate(rows):
            if r0 <= r < r1:
                sel = cols < r
                off = _pairs_before(r0, int(r))
                assert np.array_equal(host[off + cols[sel]].astype(np.int64), ref[:, ri, sel].T), int(r)
                checked += 1
        assert checked >= 2


# ------------------------------------------------------------------------------- 2. launches, buffers and streams
N_MULTI = 20_000  # not a multiple of 128, 80 or 640
CAP_MULTI = 4096
HOST_FIRST = 10_000  # one host call: 4,096 + 4,096 + 1,808 variants, alternating the two stage buffers
DEVICE_COMPLETE = (6_000, 4_096, 2_500)  # complete=True calls from one buffer, each overwritten right after the call
DEVICE_ORDERED = 3_000  # complete=False: written on the context's stream just before the call
TOTAL_MULTI = HOST_FIRST + sum(DEVICE_COMPLETE) + DEVICE_ORDERED + 1
BLOCK = 2500


def _feed_ts_sequence(ctx, job, full, host):
    """The TS call sequence: host add, device adds whose buffer is rewritten on the context's stream after each call,
    a device add whose source that stream writes just before the call, and one single-variant add."""
    import torch

    row_bytes = full.shape[1]
    job.add_variants(host[:HOST_FIRST])
    ext = torch.cuda.ExternalStream(ctx.stream(), device=full.device)
    buf = torch.full((max(DEVICE_COMPLETE + (DEVICE_ORDERED,)), row_bytes), 0xFF, dtype=torch.uint8, device=full.device)
    buf[: DEVICE_COMPLETE[0]] = full[HOST_FIRST : HOST_FIRST + DEVICE_COMPLETE[0]]
    torch.cuda.synchronize()
    off = HOST_FIRST
    sizes = list(DEVICE_COMPLETE) + [DEVICE_ORDERED]
    written = None
    for k, sz in enumerate(DEVICE_COMPLETE):
        if written is not None:
            # complete=True promises a finished source (the library's copy waits for nothing on the context's
            # stream), so the rewrite queued there after the previous call has to be done first
            written.synchronize()
        job.add_variants_device(buf.data_ptr(), row_bytes, sz, complete=True)
        off += sz
        with torch.cuda.stream(ext):  # allowed: work queued on the context's stream after the call, no sync in between
            buf[: sizes[k + 1]].copy_(full[off : off + sizes[k + 1]])
            written = torch.cuda.Event()
            written.record()
    # still queued on the context's stream: exactly what complete=False (ordered on that stream) is for
    job.add_variants_device(buf.data_ptr(), row_bytes, DEVICE_ORDERED, complete=False)
    off += DEVICE_ORDERED
    with torch.cuda.stream(ext):
        buf.fill_(0xFF)  # again after the call: must not reach the copy above
    job.add_variants(host[off : off + 1])
    assert off + 1 == TOTAL_MULTI
    ctx.synchronize()
    del buf


def _device_counts(job, r0, r1):
    import torch

    out = torch.empty(_pairs_before(r0, r1) * 5, dtype=torch.int32, device="cuda")
    job.counts_to_device(out.data_ptr(), r0, r1)
    job.ctx.synchronize()
    return out


@pytest.mark.gpu
def test_king_ts_multi_launch_and_stream_order(gpu_ctx):
    """20,000 samples (19,750 TS tiles, many waves of two CTAs per SM) with a 4,096-variant stage cap: host,
    complete and stream-ordered device sources, and a single variant, against the popcount kernel (96-column tiles,
    one staged block, no double buffering) fed the same variants from the host, over the whole triangle; a sampled
    set of pairs against the exact reference; and a row block that is not tile-aligned against the full job."""
    import torch

    from bench import synth_genovecs

    dev = torch.device("cuda", 0)
    full = synth_genovecs(torch, N_MULTI, 0, TOTAL_MULTI, dev, seed=4242)
    torch.cuda.synchronize()
    host = full.cpu().numpy().view(np.uint64)
    with KingJob(gpu_ctx, N_MULTI, 0, N_MULTI, KING_ALGO_TENSOR_TS, max_variants_per_add=CAP_MULTI) as ts, KingJob(gpu_ctx, N_MULTI, 0, N_MULTI, KING_ALGO_POPCOUNT) as pc:
        _feed_ts_sequence(gpu_ctx, ts, full, host)
        pc.add_variants(host)
        assert int(lib.pl2gpu_king_variants_added(ts._h)) == TOTAL_MULTI == int(lib.pl2gpu_king_variants_added(pc._h))
        for r0 in range(0, N_MULTI, BLOCK):
            a, b = _device_counts(ts, r0, r0 + BLOCK), _device_counts(pc, r0, r0 + BLOCK)
            assert torch.equal(a, b), f"rows [{r0}, {r0 + BLOCK}): TS differs from popcount at {int((a != b).sum())} of {a.numel()} words"
            del a, b

        rng = np.random.default_rng(5)
        rows = np.unique(np.concatenate([[1, 127, 128, 7777, 7776, 19_996, 19_999, 19_200, 19_839], rng.choice(np.arange(2, N_MULTI), size=23, replace=False)]))
        cols = np.unique(np.concatenate([[0, 79, 80, 7775, 19_198, 19_199, 19_998], rng.choice(N_MULTI, size=2048, replace=False)]))
        ref = king_ref_counts(_sample_codes(full, rows), _sample_codes(full, cols))
        for ri, r in enumerate(rows):
            sel = cols < r
            assert np.array_equal(ts.counts(int(r), int(r) + 1)[cols[sel]].astype(np.int64), ref[:, ri, sel].T), int(r)

        r0, r1 = 7_777, 19_997
        with KingJob(gpu_ctx, N_MULTI, r0, r1, KING_ALGO_TENSOR_TS, max_variants_per_add=CAP_MULTI) as part:
            _feed_ts_sequence(gpu_ctx, part, full, host)
            for b0 in range(r0, r1, BLOCK):
                b1 = min(r1, b0 + BLOCK)
                a, b = _device_counts(part, b0, b1), _device_counts(ts, b0, b1)
                assert torch.equal(a, b), f"row block [{r0}, {r1}) differs from the full job in rows [{b0}, {b1})"
                del a, b
