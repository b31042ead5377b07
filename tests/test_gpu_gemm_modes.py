"""Every launch mode of the DMMA GEMM (csrc/dgemm_nt.cuh) against a NumPy model of its documented semantics, one case
per call site at that call site's own descriptor pattern, through ace_dbg_gemm_nt_desc.

Operands are small integers (|x| <= 255, K <= 8192) and alpha, beta are 1, -1, 2 / 0, 1/2, 1, so every sum is exact
in FP64 in any order and the GPU must equal the model bit for bit.  The model also records which elements the launch
may read and write: every other element of every buffer is NaN, so a wrong k trim, diagonal-tile redirect, stride or
tile decode reads a NaN (or a wrong value), and a stray store overwrites a NaN."""
import zlib

import numpy as np
import pytest

from additivecausalexpansion_b200 import api

pytestmark = pytest.mark.gpu

TB, BM, BN, GROUP = 128, 128, 64, 8


# ----------------------------------------------------------------------------------------------- the model
def tile_list(d):
    """(ti, tj) of every tile the launch computes, in its linear order L: group rasterisation, or lower_only rows of
    2*ti + 2 tiles; with tile_stride > 1 only L = tile_first + q * tile_stride."""
    M, N = d["M"], d["N"]
    if d.get("lower_only"):
        T = M // BM
        tiles = T * (T + 1)
    else:
        tiles = (M // BM) * (N // BN)
    stride, first = d.get("tile_stride", 0), d.get("tile_first", 0)
    out = []
    for L in (range(first, tiles, stride) if stride > 1 else range(tiles)):
        if d.get("lower_only"):
            t = int((np.sqrt(4.0 * L + 1.0) - 1.0) * 0.5)
            while t * (t + 1) > L:
                t -= 1
            while (t + 1) * (t + 2) <= L:
                t += 1
            out.append((t, L - t * (t + 1)))
        else:
            tiles_m, tiles_n = M // BM, N // BN
            per_group = GROUP * tiles_n
            first_m = (L // per_group) * GROUP
            gsize = min(GROUP, tiles_m - first_m)
            r = L % per_group
            out.append((first_m + r % gsize, r // gsize))
    return out


def gemm_nt_ref(d, bufs, track=False):
    """C = beta*C + alpha*A*B^T as one launch of the descriptor d on the flat buffers bufs (pointer fields are
    (buffer, offset) pairs).  Returns the buffers after the launch; with track=True instead (reads, writes): one
    boolean mask per buffer of the elements the launch reads / stores."""
    out = [b.copy() for b in bufs]
    rd = [np.zeros(b.size, bool) for b in bufs]
    wr = [np.zeros(b.size, bool) for b in bufs]
    M, K = d["M"], d["K"]
    alpha, beta = d.get("alpha", 1.0), d.get("beta", 0.0)
    ks = d.get("ksplit", 0) if d.get("ksplit", 0) > 1 else 1
    batch = max(1, d.get("batch", 0))
    r128, c64 = np.arange(BM), np.arange(BN)
    tiles = tile_list(d)

    def ptr(name, q):
        b, off = d[name]
        stride = d.get("s" + name, 0)
        return b, off + q * stride

    for qe in range(batch * ks):
        q, chunk = (qe // ks, qe % ks) if ks > 1 else (qe, 0)
        bA, oA = ptr("A", q)
        bB, oB = ptr("B", q)
        bC, oC = ptr("C", qe)
        for ti, tj in tiles:
            i0, j0 = ti * BM, tj * BN
            if i0 >= M - q * d.get("m_dec", 0):
                continue
            a_off = d.get("a_row_off", 0) + q * d.get("s_row_off", 0)
            tia = ti + a_off // TB
            kb, ke = 0, K
            if d.get("a_tri") == 1:
                kb = i0 + a_off
            if d.get("a_tri") == 2:
                ke = i0 + a_off + BM
            if d.get("b_tri") == 2:
                ke = min(ke, (j0 // TB + 1) * TB)
            if ks > 1:
                kb, ke = max(kb, chunk * d["klen"]), min(ke, (chunk + 1) * d["klen"])
            acc = np.zeros((BM, BN))
            for k0 in range(kb, ke, TB):
                kk = np.arange(TB)
                if "Adiag" in d and k0 // TB == tia:
                    b, o = ptr("Adiag", q)
                    ia = o + tia * TB * TB + kk[None, :] * TB + r128[:, None]
                else:
                    b, o = bA, oA
                    ia = o + i0 + r128[:, None] + (k0 + kk[None, :]) * d["lda"]
                A = bufs[b][ia]
                rd[b][ia] = True
                jb = j0 // TB
                if "Bdiag" in d and k0 // TB == jb:
                    b, o = ptr("Bdiag", q)
                    ib = o + jb * TB * TB + kk[None, :] * TB + j0 % TB + c64[:, None]
                else:
                    b, o = bB, oB
                    ib = o + j0 + c64[:, None] + (k0 + kk[None, :]) * d["ldb"]
                B = bufs[b][ib]
                rd[b][ib] = True
                acc += A @ B.T
            ic = oC + (i0 + r128[:, None]) + (j0 + c64[None, :]) * d["ldc"]
            if beta != 0.0:
                res = beta * bufs[bC][ic] + alpha * acc
                rd[bC][ic] = True
            else:
                res = alpha * acc
            out[bC][ic] = res
            wr[bC][ic] = True
            if "Ct" in d:
                bT, oT = ptr("Ct", qe)
                it = oT + (j0 + c64[None, :]) + (i0 + r128[:, None]) * d["ldct"]
                out[bT][it] = res
                wr[bT][it] = True
    return (rd, wr) if track else out


def make_bufs(d, lens, rng, ints=True):
    """Buffers for the descriptor: the elements the model reads get values (integers in [-255, 255], or normals),
    everything else is NaN."""
    probe = [np.zeros(n) for n in lens]
    rd, _ = gemm_nt_ref(d, probe, track=True)
    bufs = []
    for n, m in zip(lens, rd):
        b = np.full(n, np.nan)
        v = rng.integers(-255, 256, size=n).astype(np.float64) if ints else rng.standard_normal(n)
        b[m] = v[m]
        bufs.append(b)
    return bufs


def launch(d, bufs):
    got, status = api.dbg_gemm_nt_desc(d, bufs)
    assert status == 0, status
    return got


def run_case(d, lens, seed, ints=True):
    rng = np.random.default_rng(seed)
    bufs = make_bufs(d, lens, rng, ints)
    got = launch(d, bufs)
    ref = gemm_nt_ref(d, bufs)
    for b, (g, r) in enumerate(zip(got, ref)):
        if ints:
            assert np.array_equal(g, r, equal_nan=True), (b, np.flatnonzero(~((g == r) | (np.isnan(g) & np.isnan(r))))[:8])
        else:
            assert np.array_equal(np.isnan(g), np.isnan(r)), b
            ok = ~np.isnan(r)
            assert np.abs(g[ok] - r[ok]).max(initial=0.0) <= 1e-12 * d["K"], b
    _, wr = gemm_nt_ref(d, bufs, track=True)
    assert any(m.any() for m in wr)  # the case stores something
    return got, ref


# ----------------------------------------------------------------------------------------------- call-site cases
def sq(nb):
    return nb * TB, (nb * TB) ** 2  # ld and length of an nb x nb block matrix


def tiles_of(nb):
    return nb * TB * TB  # length of nb diagonal 128 x 128 tiles


def blk(ld, rb, cb):
    return rb * TB + cb * TB * ld


def case_upd_a():
    # chol.cuh upd_a: rows [j1, nb) x cols [j1, j2) of A -= panel * panel^T
    nb, j0, j1, j2 = 11, 0, 4, 8
    ld, n = sq(nb)
    d = dict(A=(0, blk(ld, j1, j0)), lda=ld, B=(0, blk(ld, j1, j0)), ldb=ld, C=(0, blk(ld, j1, j1)), ldc=ld,
             M=(nb - j1) * TB, N=(j2 - j1) * TB, K=(j1 - j0) * TB, alpha=-1.0, beta=1.0)
    return d, [n]


def case_upd_b():
    # chol.cuh upd_b: lower tiles of the square block [j2, nb)
    nb, j0, j1, j2 = 14, 0, 4, 8
    ld, n = sq(nb)
    d = dict(A=(0, blk(ld, j2, j0)), lda=ld, B=(0, blk(ld, j2, j0)), ldb=ld, C=(0, blk(ld, j2, j2)), ldc=ld,
             M=(nb - j2) * TB, N=(nb - j2) * TB, K=(j1 - j0) * TB, alpha=-1.0, beta=1.0, lower_only=1)
    return d, [n]


def case_panel_trsm():
    # chol.cuh:437 fused panel TRSM: Wp[j1:] = A[j1:, J] * X_JJ^T, X_JJ lower (b_tri 2) with DX diagonal tiles
    nb, j0, j1 = 13, 4, 8
    ld, n = sq(nb)
    d = dict(A=(0, blk(ld, j1, j0)), lda=ld, B=(0, blk(ld, j0, j0)), ldb=ld, b_tri=2, Bdiag=(1, j0 * TB * TB),
             C=(2, j1 * TB), ldc=ld, M=(nb - j1) * TB, N=(j1 - j0) * TB, K=(j1 - j0) * TB, alpha=1.0, beta=0.0)
    return d, [n, tiles_of(nb), ld * (j1 - j0) * TB]


def case_incr_first():
    # chol.cuh:463 incremental inverse, Wt = U[0:j0, 0:j0] * L[J, 0:j0]^T (a_tri 1, DU diagonal tiles) into Bf
    nb, j0, j1 = 14, 12, 14
    ld, n = sq(nb)
    s1, s2 = j0 * TB, (j1 - j0) * TB
    d = dict(A=(0, 0), lda=ld, a_tri=1, Adiag=(1, 0), B=(0, blk(ld, j0, 0)), ldb=ld, C=(2, 0), ldc=s1,
             M=s1, N=s2, K=s1, alpha=1.0, beta=0.0)
    return d, [n, tiles_of(nb), n]


def case_incr_second():
    # chol.cuh:469 X[J, 0:j0] = -X_JJ * Wt^T (a_tri 2, DX tiles) with the transposed copy U[0:j0, J]
    nb, j0, j1 = 14, 12, 14
    ld, n = sq(nb)
    s1, s2 = j0 * TB, (j1 - j0) * TB
    d = dict(A=(0, blk(ld, j0, j0)), lda=ld, a_tri=2, Adiag=(1, j0 * TB * TB), B=(2, 0), ldb=s1,
             C=(0, blk(ld, j0, 0)), ldc=ld, Ct=(0, blk(ld, 0, j0)), ldct=ld, M=s2, N=s1, K=s2, alpha=-1.0, beta=0.0)
    return d, [n, tiles_of(nb), n]


def _trtri(nb, h, q0, cnt, s2, second):
    # chol.cuh trtri_level: node q = q0 .. q0+cnt-1 of level h, regular nodes batched with node strides
    ld, n = sq(nb)
    s1 = h * TB
    a = q0 * 2 * h
    c = a + h
    node = 2 * h * TB * (ld + 1)
    ws = q0 * s1 * s1
    if not second:
        d = dict(A=(0, blk(ld, a, a)), lda=ld, a_tri=1, Adiag=(1, a * TB * TB), B=(0, blk(ld, c, a)), ldb=ld,
                 C=(2, ws), ldc=s1, M=s1, N=s2, K=s1, alpha=1.0, beta=0.0)
        if cnt > 1:
            d.update(batch=cnt, sA=node, sB=node, sC=s1 * s1, sAdiag=2 * h * TB * TB)
    else:
        d = dict(A=(0, blk(ld, c, c)), lda=ld, a_tri=2, Adiag=(1, c * TB * TB), B=(2, ws), ldb=s1,
                 C=(0, blk(ld, c, a)), ldc=ld, Ct=(0, blk(ld, a, c)), ldct=ld, M=s2, N=s1, K=s2, alpha=-1.0, beta=0.0)
        if cnt > 1:
            d.update(batch=cnt, sA=node, sB=s1 * s1, sC=node, sCt=node, sAdiag=2 * h * TB * TB)
    return d, [n, tiles_of(nb), n]


def case_uut():
    # chol.cuh uut_inverse (DMMA): K^-1 = U U^T, lower tiles with the mirrored copy into the same buffer
    nb = 9
    ld, n = sq(nb)
    d = dict(A=(0, 0), lda=ld, a_tri=1, Adiag=(1, 0), B=(0, 0), ldb=ld, Bdiag=(1, 0), C=(2, 0), ldc=ld,
             Ct=(2, 0), ldct=ld, M=nb * TB, N=nb * TB, K=nb * TB, alpha=1.0, beta=0.0, lower_only=1)
    return d, [n, tiles_of(nb), n]


def case_chain():
    # shard_dense.cuh chain_gemm of the head TRSM (b_tri 2 + Bdiag): split over K into 128-chunks, partials in ws
    nb, j0, j1 = 12, 4, 8
    ld, n = sq(nb)
    M, N, K = (nb - j1) * TB, (j1 - j0) * TB, (j1 - j0) * TB
    d = dict(A=(0, blk(ld, j1, j0)), lda=ld, B=(0, blk(ld, j0, j0)), ldb=ld, b_tri=2, Bdiag=(1, j0 * TB * TB),
             C=(2, 0), ldc=M, M=M, N=N, K=K, alpha=1.0, beta=0.0, ksplit=K // TB, klen=TB, sA=0, sB=0, sC=M * N)
    return d, [n, tiles_of(nb), M * N * (K // TB)]


def case_shard_incr_first(cf=0):
    # shard_dense.cuh:362: Wt_c = U[c rows, 0:j0] * L[J, 0:j0]^T for a rank's panels c = cf, cf + G, ... (a_tri 1 on a
    # row slice, batched over the panels, split-K into 2048-chunks with K = j0 * 128 not a multiple of 2048)
    G, pb, J = 2, 4, 5
    j0, j1 = J * pb, J * pb + pb
    ld = j1 * TB
    pw, step, wJ, KL = pb * TB, G * pb * TB, (j1 - j0) * TB, 2048
    K = j0 * TB
    S = (K + KL - 1) // KL
    cnt = (J - cf + G - 1) // G
    length = pw * wJ
    d = dict(A=(0, cf * pw), lda=ld, a_tri=1, a_row_off=cf * pw, s_row_off=step, Adiag=(1, 0), B=(0, blk(ld, j0, 0)),
             ldb=ld, C=(2, 0), ldc=pw, M=pw, N=wJ, K=K, alpha=1.0, beta=0.0, batch=cnt, sA=step, sB=0, sC=length,
             ksplit=S, klen=KL)
    return d, [ld * K, tiles_of(j1), length * cnt * S]


def case_shard_incr_second():
    # shard_dense.cuh:384: X[J, c] = -X_JJ * Wt_c^T for the panels of rank cf, batched dual store (sA = 0)
    G, pb, J, nb, cf = 2, 4, 3, 14, 0
    j0 = J * pb
    ld, n = sq(nb)
    pw, step, wJ = pb * TB, G * pb * TB, (nb - j0) * TB
    cnt = (J - cf + G - 1) // G
    d = dict(A=(0, blk(ld, j0, j0)), lda=ld, a_tri=2, Adiag=(1, j0 * TB * TB), B=(2, 0), ldb=pw,
             C=(0, blk(ld, j0, cf * pb)), ldc=ld, Ct=(0, blk(ld, cf * pb, j0)), ldct=ld, M=wJ, N=pw, K=wJ,
             alpha=-1.0, beta=0.0, batch=cnt, sA=0, sB=pw * wJ, sC=step * ld, sCt=step)
    return d, [n, tiles_of(nb), pw * wJ * cnt]


def case_shard_apply():
    # shard_dense.cuh:409: a rank's panels c, c + G, ... of A -= pan pan^T in one batch of shrinking height (m_dec)
    G, pb, nb, c, cnt = 2, 2, 14, 2, 3
    j2 = c * pb
    ld, n = sq(nb)
    c0 = c * pb
    mB, wJ, step = (nb - j2) * TB, 2 * TB, G * pb * TB
    d = dict(A=(1, (c0 - j2) * TB), lda=mB, B=(1, (c0 - j2) * TB), ldb=mB, C=(0, blk(ld, c0, c0)), ldc=ld,
             M=(nb - c0) * TB, N=pb * TB, K=wJ, alpha=-1.0, beta=1.0, batch=cnt, sA=step, sB=step, sC=step * (ld + 1),
             m_dec=step)
    return d, [n, mB * wJ]


def case_trtri_sharded(second=False, ro_slice=3):
    # shard_dense.cuh trtri_level_sharded, node (a, c) = (8, 12) of level h = 4 split over G = 2 ranks (4 slices of
    # 128 rows): the first product on a row slice of U11 (pointer offset + a_row_off, Adiag of the node), the second
    # into the node's columns of X21 with the transposed copy packed into the staging chunk
    G, h, a, nb = 2, 4, 8, 15
    c = a + h
    hs = h // (2 * G)
    Rs, s1 = hs * TB, h * TB
    s2 = min(h, nb - c) * TB
    ld, n = sq(nb)
    ro = ro_slice * Rs
    if not second:
        d = dict(A=(0, blk(ld, a, a) + ro), lda=ld, a_tri=1, a_row_off=ro, Adiag=(1, a * TB * TB),
                 B=(0, blk(ld, c, a)), ldb=ld, C=(2, 0), ldc=Rs, M=Rs, N=s2, K=s1, alpha=1.0, beta=0.0)
        return d, [n, tiles_of(nb), Rs * s2]
    d = dict(A=(0, blk(ld, c, c)), lda=ld, a_tri=2, Adiag=(1, c * TB * TB), B=(2, 0), ldb=Rs,
             C=(0, blk(ld, c, a) + ro * ld), ldc=ld, Ct=(3, 0), ldct=Rs, M=s2, N=Rs, K=s2, alpha=-1.0, beta=0.0)
    return d, [n, tiles_of(nb), Rs * s2, Rs * s2]


def case_atri2_row_slice():
    # no call site yet: the lower-triangular operand on a row slice (a_tri 2 + a_row_off), the documented k trim and
    # diagonal-tile redirect at row block ti + a_row_off / 128
    nb, c, ro = 12, 4, 3 * TB
    ld, n = sq(nb)
    s2 = (nb - c) * TB
    d = dict(A=(0, blk(ld, c, c) + ro), lda=ld, a_tri=2, a_row_off=ro, Adiag=(1, c * TB * TB), B=(2, 0), ldb=TB,
             C=(3, 0), ldc=s2 - ro, M=s2 - ro, N=TB, K=s2, alpha=-1.0, beta=0.0)
    return d, [n, tiles_of(nb), TB * s2, (s2 - ro) * TB]


def case_posterior():
    # ace_b200.cu posterior_rows_tri: T = Kx * X^T, X = L^-1 lower (b_tri 2) with DX diagonal tiles, M = nx_pad
    nx_pad, nb = 384, 10
    ld, n = sq(nb)
    d = dict(A=(0, 0), lda=nx_pad, B=(1, 0), ldb=ld, b_tri=2, Bdiag=(2, 0), C=(3, 0), ldc=nx_pad,
             M=nx_pad, N=ld, K=ld, alpha=1.0, beta=0.0)
    return d, [nx_pad * ld, n, tiles_of(nb), nx_pad * ld]


CASES = {
    "upd_a": case_upd_a,
    "upd_b_lower_only": case_upd_b,
    "panel_trsm_btri_bdiag": case_panel_trsm,
    "incr_inverse_atri1": case_incr_first,
    "incr_inverse_atri2_ct": case_incr_second,
    "trtri_level_batch_first": lambda: _trtri(11, 2, 0, 2, 2 * TB, False),
    "trtri_level_batch_second": lambda: _trtri(11, 2, 0, 2, 2 * TB, True),
    "trtri_level_ragged_first": lambda: _trtri(11, 2, 2, 1, TB, False),
    "trtri_level_ragged_second": lambda: _trtri(11, 2, 2, 1, TB, True),
    "uut_inverse_inplace": case_uut,
    "chain_gemm_splitk": case_chain,
    "shard_incr_splitk_rank0": lambda: case_shard_incr_first(0),
    "shard_incr_splitk_rank1": lambda: case_shard_incr_first(1),
    "shard_incr_dual_store": case_shard_incr_second,
    "shard_apply_m_dec": case_shard_apply,
    "trtri_sharded_slice_first": lambda: case_trtri_sharded(False, 3),
    "trtri_sharded_slice1_first": lambda: case_trtri_sharded(False, 1),
    "trtri_sharded_second": lambda: case_trtri_sharded(True, 2),
    "posterior_btri_bdiag": case_posterior,
    "atri2_row_slice": case_atri2_row_slice,
}

# beta != 0 variants where the call site has beta = 0, and alpha = 2: every value of alpha / beta once
SCALES = {"upd_a": (2.0, 0.5), "chain_gemm_splitk": (2.0, 0.0), "posterior_btri_bdiag": (-1.0, 0.5)}


@pytest.mark.parametrize("name", sorted(CASES))
def test_call_site_exact(name):
    d, lens = CASES[name]()
    run_case(d, lens, seed=zlib.crc32(name.encode()))


@pytest.mark.parametrize("name", sorted(SCALES))
def test_call_site_exact_scaled(name):
    d, lens = CASES[name]()
    d["alpha"], d["beta"] = SCALES[name]
    run_case(d, lens, seed=7)


@pytest.mark.parametrize("name", sorted(CASES))
def test_call_site_float(name):
    d, lens = CASES[name]()
    run_case(d, lens, seed=11, ints=False)


def test_uut_inverse_symmetric():
    d, lens = case_uut()
    got, _ = run_case(d, lens, seed=3)
    n = d["M"]
    C = got[2].reshape(n, n, order="F")
    assert not np.isnan(C).any()
    assert np.array_equal(C, C.T)


def test_split_k_chunks_before_k_begin_store_zeros():
    d, lens = case_shard_incr_first(0)
    got, _ = run_case(d, lens, seed=5)
    # panel 4 (problem q = 2) starts at row 2048 = k_begin of its tiles: chunk 0 [0, 2048) lies wholly before it
    pw, wJ = d["M"], d["N"]
    part = got[2].reshape(-1, pw * wJ)  # entry qe = q * S + chunk
    S = d["ksplit"]
    assert S == 2 and d["K"] % d["klen"] != 0
    assert np.array_equal(part[2 * S + 0], np.zeros(pw * wJ))
    assert np.isfinite(part[2 * S + 1]).all() and np.any(part[2 * S + 1] != 0)


def test_m_dec_tail_untouched():
    """Problem q = 1 of the shrinking batch starts at block (8, 8) with 6 block rows: the rows its tiles would cover
    without the m_dec exit lie past the matrix and wrap into the top rows of the next columns, which stay NaN."""
    d, lens = case_shard_apply()
    got, _ = run_case(d, lens, seed=9)
    ld = int(round(np.sqrt(lens[0])))
    A = got[0].reshape(ld, ld, order="F")
    assert np.isnan(A[:4 * TB, 8 * TB + 1:10 * TB + 1]).all()
    assert np.isfinite(A[8 * TB:, 8 * TB:10 * TB]).all()
    no_exit = gemm_nt_ref(dict(d, m_dec=0), [np.zeros(2 * n) for n in lens], track=True)[1][0][:lens[0]]
    assert no_exit.reshape(ld, ld, order="F")[:4 * TB, 8 * TB + 1:10 * TB + 1].any()


@pytest.mark.parametrize("world", range(1, 9))
def test_uut_tile_subsets_partition_lower_only(world):
    """uut_inverse_sharded: ranks r = 0..world-1 with tile_first = r, tile_stride = world, each into its own NaN C,
    every result equal to the model, in place (Ct == C) as the call site runs it.  With the transposed copy in a
    buffer of its own, the C stores of the ranks are disjoint and together exactly the lower_only tiles, and so are
    the Ct stores."""
    d, lens = case_uut()
    sep = dict(d, Ct=(3, 0))
    lens4 = lens + [lens[2]]
    full = gemm_nt_ref(sep, [np.zeros(n) for n in lens4], track=True)[1]
    seen_c, seen_t = np.zeros(lens[2], int), np.zeros(lens[2], int)
    base = make_bufs(sep, lens4, np.random.default_rng(world))
    for r in range(world):
        for dr, bufs in ((dict(d, tile_first=r, tile_stride=world), base[:3]),
                         (dict(sep, tile_first=r, tile_stride=world), base)):
            got = launch(dr, bufs)
            ref = gemm_nt_ref(dr, bufs)
            for g, f in zip(got, ref):
                assert np.array_equal(g, f, equal_nan=True), (r, len(bufs))
        seen_c += ~np.isnan(got[2])
        seen_t += ~np.isnan(got[3])
    assert seen_c.max() == 1 and seen_t.max() == 1
    assert np.array_equal(seen_c == 1, full[2]) and np.array_equal(seen_t == 1, full[3])


# ----------------------------------------------------------------------------------------------- rejections
@pytest.mark.parametrize("bad", ["M", "N", "K", "tile_first", "tile_batch", "klen_unaligned", "klen_zero",
                                 "a_row_off", "s_row_off"])
def test_launcher_rejects(bad):
    n = 256 * 256
    d = dict(A=(0, 0), lda=256, B=(0, 0), ldb=256, C=(1, 0), ldc=256, M=256, N=256, K=256, alpha=1.0, beta=0.0)
    d.update({"M": dict(M=192), "N": dict(N=192), "K": dict(K=200), "tile_first": dict(tile_first=3, tile_stride=3),
              "tile_batch": dict(tile_first=0, tile_stride=2, batch=2), "klen_unaligned": dict(ksplit=2, klen=100),
              "klen_zero": dict(ksplit=2, klen=0), "a_row_off": dict(a_tri=1, a_row_off=64),
              "s_row_off": dict(a_tri=1, batch=2, s_row_off=64)}[bad])
    bufs = [np.ones(n), np.full(n, np.nan)]
    got, status = api.dbg_gemm_nt_desc(d, bufs)
    assert status == -2, status
    # nothing was launched: C comes back as it went (the hook downloads the buffers after a refusal too)
    assert np.isnan(got[1]).all() and np.array_equal(got[0], bufs[0])


@pytest.mark.parametrize("short", ["A", "B", "C", "Ct", "Adiag", "m_dec"])
def test_hook_refuses_operands_outside_their_buffers(short):
    """A descriptor that reaches one element past the end of a buffer is refused (ACE_ERR_USAGE) before any device
    work, and so is a shrinking batch without its m_dec exit, whose last problems run past the end of A."""
    case, buf = {"A": (case_posterior, 0), "B": (case_posterior, 1), "C": (case_posterior, 3),
                 "Ct": (lambda: case_trtri_sharded(True, 2), 3), "Adiag": (case_uut, 1),
                 "m_dec": (case_shard_apply, None)}[short]
    d, lens = case()
    if short == "m_dec":
        d = dict(d, m_dec=0)
    else:
        lens[buf] -= 1
    bufs = [b[:n] for b, n in zip(make_bufs(d, [2 * n for n in lens], np.random.default_rng(1)), lens)]
    got, status = api.dbg_gemm_nt_desc(d, bufs)
    assert status == -1, (short, status)
    assert all(np.array_equal(g, b, equal_nan=True) for g, b in zip(got, bufs))
