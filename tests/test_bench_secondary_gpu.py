"""The secondary kernels bench.py reports (grm_ts_kernel, ld_ts_kernel, score_kernel) at the benchmark's shapes,
through the calls it makes, against exact or fp64 references on sampled outputs.

The GRM reference (`grm_rows_ref`) restates oracle.grm for a few rows against every sample, in fp64 on the
device: oracle.grm itself forms the whole N x N product on the host, which at 16,384 samples x 262,144 variants
is out of reach.  Entry (i, j) of oracle.grm with given REF frequencies depends only on samples i and j, so rows of
a subset are rows of the whole; test_grm_rows_ref_matches_oracle checks both on the host."""
import ctypes as C

import numpy as np
import pytest

from oracle import plink_oracle as orc
from plink_ng_b200.capi import check, lib
from plink_ng_b200.host import GrmJob

RTOL, ATOL = 1e-5, 1e-10  # the GRM contract of tests/test_grm_gpu.py


def _unpack(g, n):
    """Codes uint8 [variants, n] of a device genovec tensor g = uint8 [variants, row_bytes] (PgrGet layout)."""
    import torch

    return torch.stack([(g >> s) & 3 for s in (0, 2, 4, 6)], dim=-1).reshape(g.shape[0], -1)[:, :n]


def _pack_mask(mask, row_bytes):
    """bool [variants, n] -> uint8 [variants, row_bytes] with both bits of every selected sample set."""
    import torch

    m = torch.zeros((mask.shape[0], row_bytes * 4), dtype=torch.uint8, device=mask.device)
    m[:, : mask.shape[1]] = mask.to(torch.uint8) * 3
    q = m.view(mask.shape[0], row_bytes, 4)
    return q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)


def grm_rows_ref(codes_r, codes_c, ref_freq, chunk=8192):
    """oracle.grm restated for row samples R against column samples C: (G [|R|, |C|] float64, obs [|R|, |C|] int64
    or None) from codes [variants, |R|] and [variants, |C|] and the REF frequencies [variants] (all of them with
    2 f (1 - f) above 2^-44).  numpy on the host or torch on the tensors' device, fp64 throughout; the division
    by the per-pair observation count (or by the variant count when no call is missing) is oracle.grm's."""
    torch_in = not isinstance(codes_r, np.ndarray)
    if torch_in:
        import torch

        xp, f64, asf = torch, (lambda x: x.to(torch.float64)), (lambda x: torch.as_tensor(x, dtype=torch.float64, device=codes_r.device))
    else:
        xp, f64, asf = np, (lambda x: x.astype(np.float64)), (lambda x: np.asarray(x, dtype=np.float64))
    ref_freq = np.asarray(ref_freq, dtype=np.float64)
    alt = 1.0 - ref_freq
    slope = 1.0 / np.sqrt(2 * ref_freq * alt)
    icpt = -2 * alt * slope
    table = np.stack([icpt, icpt + slope, icpt + 2 * slope, np.zeros_like(slope)], axis=1)  # centered_varmaj
    g = mr = mc = both = None
    for v0 in range(0, codes_r.shape[0], chunk):
        a, b = codes_r[v0 : v0 + chunk], codes_c[v0 : v0 + chunk]
        t = asf(table[v0 : v0 + chunk])
        za = _take(xp, t, a)
        zb = _take(xp, t, b)
        ma, mb = f64(a == 3), f64(b == 3)
        parts = (za.T @ zb, ma.sum(0), mb.sum(0), ma.T @ mb)
        g, mr, mc, both = parts if g is None else (g + parts[0], mr + parts[1], mc + parts[2], both + parts[3])
    if torch_in:
        g, mr, mc, both = (x.cpu().numpy() for x in (g, mr, mc, both))
    m = codes_r.shape[0]
    if not (mr.any() or mc.any()):
        return g * (1.0 / float(m)), None
    obs = m - np.rint(mr).astype(np.int64)[:, None] - np.rint(mc).astype(np.int64)[None, :] + np.rint(both).astype(np.int64)
    return g / obs.astype(np.float64), obs


def _take(xp, table, codes):
    """table [variants, 4] indexed by codes [variants, k] -> [variants, k]."""
    if xp is np:
        return np.take_along_axis(table, codes.astype(np.int64), axis=1)
    import torch

    return torch.gather(table, 1, codes.long())


def test_grm_rows_ref_matches_oracle():
    """The restatement against oracle.grm, and oracle.grm on a subset of samples against the same rows of the whole
    (with fixed REF frequencies, every entry depends on its two samples only), with and without missing calls."""
    rng = np.random.default_rng(11)
    m, n = 700, 90
    freq = rng.uniform(0.05, 0.95, size=(m, 1))
    geno = ((rng.random((m, n)) < freq).astype(np.uint8) + (rng.random((m, n)) < freq).astype(np.uint8))
    rf = rng.uniform(0.05, 0.95, size=m)
    for miss in (0.03, 0.0):
        gm = geno.copy()
        gm[rng.random((m, n)) < miss] = 3
        want, obs = orc.grm(gm, ref_freq=rf)
        sub = np.array([0, 5, 17, 40, 41, 89])
        got, got_obs = grm_rows_ref(gm[:, sub], gm, rf, chunk=128)
        assert np.allclose(got, want[sub], rtol=1e-13, atol=1e-15)
        assert (got_obs is None) == (obs is None) and (obs is None or np.array_equal(got_obs, obs[sub]))
        want_sub, obs_sub = orc.grm(gm[:, sub], ref_freq=rf)
        assert np.allclose(want_sub, want[np.ix_(sub, sub)], rtol=1e-13, atol=1e-15)
        assert obs is None or np.array_equal(obs_sub, obs[np.ix_(sub, sub)])


@pytest.mark.gpu
def test_grm_bench_shape(gpu_ctx):
    """16,384 samples, four add_variants_device calls of 65,536 distinct variants each with the bench's kind of REF
    frequencies: 40 sampled rows in full (the last row, row 0, the diagonal of each), observation counts exact."""
    import torch

    from bench import synth_genovecs

    n, m, calls = 16_384, 65_536, 4
    dev = torch.device("cuda", 0)
    rf = np.random.default_rng(0).uniform(0.05, 0.95, size=calls * m)  # the first 65,536 are the bench's
    rng = np.random.default_rng(3)
    rows = np.unique(np.concatenate([[0, 1, 127, 128, 639, 640, 8191, 16_382, n - 1], rng.choice(n, size=31, replace=False)]))
    with GrmJob(gpu_ctx, n) as job:
        gs = []
        for k in range(calls):
            g = synth_genovecs(torch, n, k * m, (k + 1) * m, dev)
            torch.cuda.synchronize()
            job.add_variants_device(g.data_ptr(), g.shape[1], m, ref_freqs=rf[k * m : (k + 1) * m])
            gs.append(g)
        gpu_ctx.synchronize()
        assert int(lib.pl2gpu_grm_variants_added(job._h)) == calls * m
        codes = torch.cat([_unpack(g, n) for g in gs])
        del gs
        want, want_obs = grm_rows_ref(codes[:, torch.as_tensor(rows, device=dev)], codes, rf)
        del codes
        assert want_obs is not None
        for ri, r in enumerate(rows):
            r = int(r)
            got, got_obs = job.rows(r, r + 1, with_obs=True)
            a, b = got[0, : r + 1], want[ri, : r + 1]
            err = np.abs(a - b)
            assert np.all(err <= RTOL * np.abs(b) + ATOL), (r, float(err.max()))
            assert np.array_equal(got_obs[0, : r + 1], want_obs[ri, : r + 1].astype(np.float32)), r


def _ld_plant(g, nf, seed=7):
    """Linkage on the device, in place: in every block of 64 variants, each later variant copies the block's first
    variant (its "hub", 1 to 63 variants earlier) for a fraction of the founders drawn from U(0.5, 1) and keeps its
    own genotypes for the others.  Variants that copy the same hub are correlated with each other and with it; the
    r^2 of such pairs spreads across 0.2 (median about 0.25), and variants of different blocks stay unlinked."""
    import torch

    gen = torch.Generator(device=g.device)
    gen.manual_seed(seed)
    mv, row_bytes = g.shape
    orig = g.clone()
    for v0 in range(0, mv, 2048):
        v1 = min(mv, v0 + 2048)
        v = torch.arange(v0, v1, device=g.device)
        hub = v // 64 * 64
        frac = torch.rand(v1 - v0, generator=gen, device=g.device) * 0.5 + 0.5
        take = (torch.rand((v1 - v0, nf), generator=gen, device=g.device) < frac[:, None]) & (v != hub)[:, None]
        mk = _pack_mask(take, row_bytes)
        g[v0:v1] = (orig[v0:v1] & ~mk) | (orig[hub] & mk)
    del orig


@pytest.mark.gpu
def test_ld_band_flags_bench_shape(gpu_ctx):
    """pl2gpu_ld_band_flags at 50,000 founders x 131,072 variants, band 499, called as bench.py calls it, with planted
    linkage: whole band rows of 48 anchors (chunk edges of the 16,384-variant launches, the first rows, the last
    variant) against the exact integer test of tests/test_ld_gpu.py."""
    import torch

    from bench import synth_genovecs

    nf, mv, band = 50_000, 131_072, 499
    thr = 0.2 * (1 + orc.SMALL_EPSILON)
    dev = torch.device("cuda", 0)
    g = synth_genovecs(torch, nf, 0, mv, dev)
    _ld_plant(g, nf)
    torch.cuda.synchronize()
    flags_t = torch.zeros((mv, band), dtype=torch.uint8).pin_memory()
    check(lib.pl2gpu_ld_band_flags(gpu_ctx.handle, C.c_void_p(g.data_ptr()), g.shape[1], nf, mv, 1, band, thr, flags_t.numpy().ctypes.data), "pl2gpu_ld_band_flags")
    flags = flags_t.numpy()
    chunk = 16_384  # variants per launch (kLdChunkVariants); each launch also re-reads the 512 variants before it
    # launch edges, row-tile (128-variant) edges after them, the first rows (band cut short by variant 0), the last
    edges = [e for k in range(1, mv // chunk) for e in (k * chunk - 1, k * chunk, k * chunk + 127, k * chunk + 128)]
    anchors = set([1, 63, 64, 127, 128, 498, 499, 500, 511, 512, 513, mv - 1] + edges)
    rng = np.random.default_rng(8)
    anchors = sorted(anchors | set(int(x) for x in rng.choice(np.setdiff1d(np.arange(band, mv), list(anchors)), size=48 - len(anchors), replace=False)))
    assert len(anchors) == 48
    n_true = n_false = n_near = 0
    for a in anchors:
        lo = max(0, a - band)
        codes = _unpack(g[lo : a + 1], nf).cpu().numpy()
        x = np.where(codes == 0, 1.0, np.where(codes == 2, -1.0, 0.0)).astype(np.float32)
        nm = (codes != 3).astype(np.float32)
        bs = np.arange(0, a - lo)
        nm_ct, s_b, q_b, s_a, q_a, dot = orc.ld_pair_components(x, nm, a - lo, bs)
        cov12 = (dot * nm_ct - s_b * s_a).astype(np.float64)
        var1 = (q_b * nm_ct - s_b * s_b).astype(np.float64)
        var2 = (q_a * nm_ct - s_a * s_a).astype(np.float64)
        want = cov12 * cov12 > thr * var1 * var2
        got = flags[a, a - lo - bs - 1].astype(bool)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"anchor {a}: flags differ for first = {(lo + bs[bad[:8]]).tolist()}"
        n_true += int(want.sum())
        n_false += int((~want).sum())
        with np.errstate(divide="ignore", invalid="ignore"):
            r2 = cov12 * cov12 / (var1 * var2)
        n_near += int((np.abs(r2 / 0.2 - 1) < 0.01).sum())
    assert n_true >= 100 and n_false >= 10_000 and n_near >= 3, (n_true, n_false, n_near)


@pytest.mark.gpu
def test_score_bench_shape(gpu_ctx):
    """pl2gpu_score_add_variants at 100,000 samples x 131,072 entries with the bench's weights and dosage codes:
    512 sampled samples (0 and 99,999 among them) against an fp64 numpy sum, dosage sums and missing counts exact."""
    import torch

    from bench import synth_genovecs

    ns, ms = 100_000, 131_072
    dev = torch.device("cuda", 0)
    g = synth_genovecs(torch, ns, 0, ms, dev)
    w4 = np.random.default_rng(2).normal(size=(ms, 4))
    d4 = np.full(ms, 0 | (1 << 2) | (2 << 4), dtype=np.uint8)
    torch.cuda.synchronize()
    h = C.c_void_p()
    check(lib.pl2gpu_score_begin(gpu_ctx.handle, ns, C.byref(h)), "pl2gpu_score_begin")
    try:
        check(lib.pl2gpu_score_add_variants(h, C.c_void_p(g.data_ptr()), g.shape[1], ms, 1, w4.ctypes.data, d4.ctypes.data), "pl2gpu_score_add_variants")
        sums = np.empty(ns)
        dos = np.empty(ns, dtype=np.uint64)
        miss = np.empty(ns, dtype=np.uint32)
        check(lib.pl2gpu_score_get(h, sums.ctypes.data, dos.ctypes.data, miss.ctypes.data), "pl2gpu_score_get")
    finally:
        lib.pl2gpu_score_end(h)
    rng = np.random.default_rng(12)
    samples = np.unique(np.concatenate([[0, 1, 31, 32, 99_968, ns - 1], rng.choice(ns, size=506, replace=False)]))
    idx = torch.as_tensor(samples, device=dev)
    codes = ((g[:, idx // 4] >> (2 * (idx % 4)).to(torch.uint8)) & 3).cpu().numpy().astype(np.int64)
    want_sum = w4[np.arange(ms)[:, None], codes].sum(axis=0)  # fp64, entry by entry
    want_dos = np.where(codes == 3, 0, codes).sum(axis=0)
    want_miss = (codes == 3).sum(axis=0)
    assert np.array_equal(dos[samples].astype(np.int64), want_dos)
    assert np.array_equal(miss[samples].astype(np.int64), want_miss)
    assert np.allclose(sums[samples], want_sum, rtol=1e-11, atol=1e-11 * np.abs(want_sum).max())
