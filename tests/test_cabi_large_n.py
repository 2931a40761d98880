"""CPU tests of the TMA SYRK work split (tlsq_plan_syrk) for every N up to the 4096-column limit: every upper 128-block
is computed exactly once, the CTA ranges are contiguous, the partial slots do not overlap, and up to N = 2048 the split
is the one the plan has always produced (which rows go into which partial sum fixes G bit for bit)."""
import ctypes

import numpy as np
import pytest

import tlsq_b200 as T

SB = 128
SMS = 148
MAX_BLK = 528          # 32 x 32 blocks of 128 columns at N = 4096
ROWS = [4096, 4400, 100_000, 1_000_018]


def plan(M, N, sms=SMS):
    lib = T.load()
    nblk, ncta, pb = ctypes.c_int(-1), ctypes.c_int(-1), ctypes.c_int64(-1)
    ns = np.full(MAX_BLK, -1, dtype=np.int32)
    cb = np.full(MAX_BLK + 1, -1, dtype=np.int32)
    po = np.full(MAX_BLK, -1, dtype=np.int32)
    vp = ctypes.c_void_p
    rc = lib.tlsq_plan_syrk(M, N, sms, ctypes.byref(nblk), ctypes.byref(ncta), ns.ctypes.data_as(vp),
                            cb.ctypes.data_as(vp), po.ctypes.data_as(vp), ctypes.byref(pb))
    assert rc == 0, lib.tlsq_last_error()
    k = nblk.value
    assert np.all(ns[k:] == -1) and np.all(cb[k + 1:] == -1) and np.all(po[k:] == -1)      # nothing written past nblk
    return k, ncta.value, ns[:k], cb[:k + 1], po[:k], pb.value


def reference_split(M, N, sms):
    """The split of syrk_tma.cu as it stood at the 2048-column limit: CTAs per block in proportion to weights 4 (off-
    diagonal) and 2.5 (diagonal), at least 1 and at most one per 32-row tile, then left-over SMs to the off-diagonal
    blocks first."""
    nb = (N + SB - 1) // SB
    nblk = nb * (nb + 1) // 2
    ntiles = (M + 31) // 32
    unit = float(sms) / (4.0 * (nblk - nb) + 2.5 * nb)
    diag = [bi == bj for bi in range(nb) for bj in range(bi, nb)]
    ns = []
    for d in diag:
        v = int((2.5 if d else 4.0) * unit)
        ns.append(min(max(v, 1), ntiles))
    total = sum(ns)
    for pas in range(4):
        if total >= sms:
            break
        for b, d in enumerate(diag):
            if total >= sms:
                break
            if (not d) == (pas % 2 == 0) and ns[b] < ntiles:
                ns[b] += 1
                total += 1
    return np.array(ns, dtype=np.int32)


@pytest.mark.parametrize("M", ROWS)
def test_syrk_plan_covers_every_upper_block_once(M):
    ntiles = (M + 31) // 32
    for N in range(65, 4097):
        nblk, ncta, ns, cb, po, pbytes = plan(M, N)
        nb = (N + SB - 1) // SB
        assert nblk == nb * (nb + 1) // 2 <= MAX_BLK
        # contiguous CTA ranges, one range per block, at least one CTA and at most one per 32-row tile
        assert cb[0] == 0 and cb[-1] == ncta
        assert np.array_equal(np.diff(cb), ns)
        assert ns.min() >= 1 and ns.max() <= ntiles
        # partial slots: disjoint ranges inside the workspace
        order = np.argsort(po, kind="stable")
        ends = po[order] + ns[order]
        assert po[order][0] >= 0 and np.all(po[order][1:] >= ends[:-1])
        assert pbytes >= int(ends.max()) * SB * SB * 8
        # the kernel's CTA -> block lookup reaches every upper block (bi <= bj) exactly once, with splits 0 .. ns-1
        cta = np.arange(ncta)
        blk = np.searchsorted(cb, cta, side="right") - 1
        split = cta - cb[blk]
        assert np.all((split >= 0) & (split < ns[blk]))
        assert np.array_equal(np.bincount(blk, minlength=nblk), ns)


@pytest.mark.parametrize("M", ROWS)
@pytest.mark.parametrize("sms", [148, 132])
def test_syrk_plan_up_to_2048_columns_is_unchanged(M, sms):
    for N in range(65, 2049):
        nblk, ncta, ns, cb, po, pbytes = plan(M, N, sms)
        ref = reference_split(M, N, sms)
        assert np.array_equal(ns, ref), N
        assert np.array_equal(cb, np.concatenate([[0], np.cumsum(ref)]))
        assert np.array_equal(po, cb[:-1])
        assert pbytes == int(ref.sum()) * SB * SB * 8


def test_syrk_plan_above_2048_columns_gives_every_block_one_cta():
    """528 blocks at N = 4096 (3.6 waves on 148 SMs): the weights put less than one CTA on every block."""
    nblk, ncta, ns, cb, po, pbytes = plan(100_000, 4096)
    assert nblk == 528 and ncta == 528 and np.all(ns == 1)
    nblk, ncta, ns, cb, po, pbytes = plan(100_000, 2049)
    assert nblk == 153 and np.all(ns == 1)


def test_syrk_plan_rejects_more_than_4096_columns():
    lib = T.load()
    i, j, p = ctypes.c_int(), ctypes.c_int(), ctypes.c_int64()
    buf = np.zeros(MAX_BLK + 1, dtype=np.int32)
    vp = buf.ctypes.data_as(ctypes.c_void_p)
    assert lib.tlsq_plan_syrk(100_000, 4097, SMS, ctypes.byref(i), ctypes.byref(j), vp, vp, vp,
                              ctypes.byref(p)) == T._cabi.TLSQ_ERR_UNSUPPORTED
    assert b"4096" in lib.tlsq_last_error()
    assert lib.tlsq_plan_syrk(0, 100, SMS, ctypes.byref(i), ctypes.byref(j), vp, vp, vp,
                              ctypes.byref(p)) == T._cabi.TLSQ_ERR_ARG
