"""Column-chunked int8-slice condensation (hb_ozaki.cu, DESIGN.md section 3.4) on a numpy model of the device order of operations:
the digits of a chunk are those of the unchunked slicing, every int32 accumulator of a chunk stays below 2^31, and the FP64 result only
differs by the grouping of the recombination sums.

The model restates the device schedule: the K stages (KS columns each) of a column chunk are split evenly over `splits` items
(hb_part_begin); an item recombines its stages in groups of chunk_stages into an FP64 partial tile (the epilogue of k_oz_gemm: the S
anti-diagonal int32 sums, smallest weight first); the first chunk writes the tile, later chunks add to it; k_oz_fixup sums the splits in
order and applies the row scales. With one chunk this is the unchunked kernel."""
import numpy as np
import pytest

from oracle import oz_model as oz


def part_begin(total, parts, p):
    return (total // parts) * p + min(p, total % parts)


def chunk_stages_for(S, KS=128):
    stages = (524288 // S) // KS
    while S * stages * KS * 4096 >= 2 ** 31:
        stages -= 1
    return stages


def gram_device_order(B, S, splits, chunk_stages, window_stages=None, KS=128):
    """C ~= B B^T in the device's order of FP64 operations. window_stages: K stages per column chunk (None: all of K, unchunked).
    Returns (C, max |int32 accumulator|, Q)."""
    M, K = B.shape
    e = oz.row_exponents(B)
    kstages = -(-K // KS)
    Q = np.zeros((S, M, kstages * KS), dtype=np.int64)
    Q[:, :, :K] = oz.slices(B, e, S)
    W = window_stages or kstages
    slot = np.zeros((splits, M, M))
    max_acc = 0
    for q, w0 in enumerate(range(0, kstages, W)):
        wst = min(W, kstages - w0)
        for s in range(splits):
            b, e2 = part_begin(wst, splits, s), part_begin(wst, splits, s + 1)
            for g0 in range(b, e2, chunk_stages):                   # one epilogue drain of TMEM
                g1 = min(g0 + chunk_stages, e2)
                Qg = Q[:, :, (w0 + g0) * KS:(w0 + g1) * KS]
                acc = np.zeros((M, M))
                for u in range(S - 1, -1, -1):                      # smallest weights first
                    T = sum(Qg[p] @ Qg[u - p].T for p in range(u + 1))
                    max_acc = max(max_acc, int(np.abs(T).max(initial=0)))
                    acc = acc + T.astype(np.float64) * 2.0 ** (-(12 + 7 * u))
                slot[s] = acc if (q == 0 and g0 == b) else slot[s] + acc
    C = np.zeros((M, M))
    for s in range(splits):
        C = C + slot[s]
    return np.ldexp(C, e[:, None] + e[None, :]), max_acc, Q


def _B(M, K, seed, decades=3.0):
    r = np.random.default_rng(seed)
    return r.standard_normal((M, K)) * 10.0 ** r.uniform(-decades, decades, size=(M, 1)) * np.sqrt(10.0 ** r.uniform(-3, 3, size=(1, K)))


def test_chunk_digits_equal_the_unchunked_digits():
    # the slicing of a column window uses the row exponents of ALL columns: its bytes are a column range of the unchunked slices
    B = _B(7, 5000, 1)
    B[2, 4100:] *= 1e6                                       # the row maximum lies in a later chunk
    e = oz.row_exponents(B)
    Q = oz.slices(B, e, 8)
    for k0 in range(0, 5000, 1280):
        Qw = oz.slices(B[:, k0:k0 + 1280], e, 8)
        np.testing.assert_array_equal(Qw, Q[:, :, k0:k0 + 1280])
    # a chunk sliced with its own row maxima would give other digits: that is what the global sweep prevents
    e_local = oz.row_exponents(B[:, :1280])
    assert not np.array_equal(oz.slices(B[:, :1280], e_local, 8), Q[:, :, :1280])


@pytest.mark.parametrize("S", [6, 7, 8])
def test_int32_accumulators_of_a_chunk_stay_below_2_31(S):
    # chunk boundaries are multiples of the recombination chunk, so an item of a chunk drains TMEM at most every chunk_stages stages:
    # the bound holds for the worst digits (all -64), and the model runs one window of the real stage count plus a ragged one
    cs = chunk_stages_for(S)
    assert S * cs * 128 * 64 * 64 < 2 ** 31
    B = -np.ones((2, cs * 128 + 300))
    C, max_acc, Q = gram_device_order(B, S, splits=1, chunk_stages=cs, window_stages=cs)
    assert max_acc < 2 ** 31
    np.testing.assert_allclose(C, B @ B.T, rtol=1e-15)


@pytest.mark.parametrize("S", [6, 7, 8])
def test_chunked_result_differs_only_at_rounding_level(S):
    # scaled-down schedule (KS = 16 columns per stage, 5 stages per recombination chunk): 4 windows of 2 recombination chunks, a ragged
    # last window shorter than `splits` stages (items with nothing to do), odd K
    B = _B(20, 16 * 5 * 2 * 3 + 16 * 2 + 7, 2 + S)
    kw = dict(S=S, splits=3, chunk_stages=5, KS=16)
    C1, acc1, Q1 = gram_device_order(B, **kw)
    Cc, accc, Qc = gram_device_order(B, window_stages=10, **kw)
    np.testing.assert_array_equal(Q1, Qc)
    assert max(acc1, accc) < 2 ** 31
    d = np.sqrt(np.outer(np.diag(C1), np.diag(C1)))
    err = (np.abs(Cc - C1) / d).max()
    assert err <= 1e-14, err
    assert np.array_equal(Cc, Cc.T)
    # and the model's unchunked order agrees with the plain slice model of oracle/oz_model.py to rounding
    C0, _ = oz.gram(B, S)
    assert (np.abs(C1 - C0) / d).max() <= 1e-14


def test_one_window_is_the_unchunked_kernel():
    B = _B(9, 16 * 23 + 5, 4)
    kw = dict(S=8, splits=4, chunk_stages=5, KS=16)
    C1, _, _ = gram_device_order(B, **kw)
    C2, _, _ = gram_device_order(B, window_stages=24, **kw)     # a window at least as long as K
    assert np.array_equal(C1, C2)
