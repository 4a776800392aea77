"""KING TS tensor kernel at the largest per-launch magnitude: one launch of 2^20 variants, with samples whose pair
counts reach 2^20, must match the popcount kernel bit for bit.  The TS kernel sums 0/+-1 products in an F32
accumulator, which is exact only while every partial sum stays below 2^24; this guards that margin."""
import numpy as np
import pytest

from plink_ng_b200.host import KING_ALGO_POPCOUNT, KING_ALGO_TENSOR_TS, KingJob

pytestmark = pytest.mark.gpu

M = 1 << 20  # kMaxStageVariantsEx: the most variants one launch accumulates
N = 640


def _genovecs():
    """[M, N / 32] uint64 genovecs (PgrGet layout: sample s at bits 2 (s % 32) of word s / 32), random codes
    except samples 0-3 all het, 4-7 all hom-REF and 8-11 all hom-ALT."""
    rng = np.random.default_rng(2024)
    by = rng.integers(0, 256, size=(M, N // 4), dtype=np.uint8)
    by[:, 0] = 0x55  # code 1 x 4
    by[:, 1] = 0x00  # code 0 x 4
    by[:, 2] = 0xAA  # code 2 x 4
    return np.ascontiguousarray(by).view("<u8").reshape(M, N // 32)


def test_king_ts_full_launch_matches_popcount(gpu_ctx):
    gv = _genovecs()
    got = {}
    for algo in (KING_ALGO_TENSOR_TS, KING_ALGO_POPCOUNT):
        with KingJob(gpu_ctx, N, 0, N, algo, max_variants_per_add=M) as job:
            job.add_variants(gv)
            got[algo] = job.counts()
    ts, pc = got[KING_ALGO_TENSOR_TS], got[KING_ALGO_POPCOUNT]
    assert ts.shape == pc.shape
    assert pc.max() >= M  # some counts do reach 2^20
    assert np.array_equal(ts, pc)
