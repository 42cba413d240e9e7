"""The fit path (assemble -> Cholesky -> triangular inverse -> K^-1 = W^T W -> gradient) at every size where its
kernel and stream schedule changes.

``schedule(N, timed)`` restates, from the sources, which schedule ``mfgp_lml_grad`` runs at N.  The GPU tests
below pick their sizes so that every schedule is reached, and ``test_gpu_cases_reach_every_schedule`` (host only)
fails when a threshold moves and a schedule is left untested:

1. Structured matrices whose factorisation is exact in FP64 in any summation order: ``mfgp_potrf``, ``mfgp_trtri``
   and ``mfgp_lauum`` must return the exact integer results, bit for bit.
2. Random GP covariances: against the NumPy oracle where it is affordable (N <= 4097), against properties, the
   cuSOLVER factor and central differences above that.
3. The timed schedule (stage events, sequential solves) against the untimed one (solves on the side stream under
   K^-1 = W^T W): same kernels on the same data, so every output must agree bit for bit.
4. The first-bad-pivot ``info`` in every schedule.
"""
import gc

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import gpy_oracle as go
from tests import util

KIND, d, E = go.KIND_COMPOSITE, 4, 1
LEAF = 128
PARTIALS = 1 << 16              # MFGP_PARTIALS, common.cuh


# ---- the schedule table -------------------------------------------------------------------------------------------
def padded(N):
    return (max(N, 1) + LEAF - 1) // LEAF * LEAF


def factor_label(npad):
    """potrf_padded + trtri_padded (mfgp_potrf / mfgp_trtri): the Cholesky driver and the inverse's form."""
    m = npad // LEAF
    if npad < 4096:                                      # LA_MIN, linalg.cu:877,972
        chol = "rec"
    else:
        chol = "la512" if npad < 24576 else "la1024"     # la_nb, linalg.cu:882
    inv = "levels" if m & (m - 1) == 0 else "rec"        # linalg.cu:1023
    return chol + "+" + inv


def schedule(N, timed):
    """Schedule of mfgp_lml_grad(_timed) at N; timed = stage events requested (h_ms != NULL)."""
    if N <= 96:                                          # MFGP_SMALL_N, capi.cu:158,393
        return "fused"
    npad = padded(N)
    label = factor_label(npad)
    nb = 512 if npad < 24576 else 1024
    if label.endswith("levels") and npad >= 8192 and (npad // 2) % nb == 0:   # linalg.cu:1041
        label = "overlap%d" % nb
    if not timed and npad >= 2048:                       # capi.cu:408
        label += "+sidesolve" if 2 * npad <= PARTIALS else "+seqsolve"
    return label


# ---- the GPU cases (module constants, so that the host test can check what they reach) ---------------------------
STRUCT_NPAD = [128, 384, 2048, 3072, 4096, 4224, 6272, 8192, 10112, 16384, 25088]
ORACLE_N = [1921, 2048, 3000, 4095, 4097]
LARGE_N = [10000, 24577, 32768, 33000]
TIMED_N = [97, 1921, 3000, 4095, 4097, 10000, 16384, 32768, 33000]
# (N, NaN rows of X, expected 1-based info)
INFO_CASES = [(50, [17], 18), (50, [49], 50), (700, [300], 301), (700, [699], 700), (3000, [1500], 1501),
              (3000, [2500, 2000], 2001), (5000, [100], 101), (5000, [511], 512), (5000, [512], 513),
              (5000, [4700], 4701), (5000, [4999], 5000), (16384, [3000], 3001), (16384, [12000], 12001),
              (16384, [9000, 8191], 8192), (24577, [13000], 13001), (24577, [24576], 24577)]
MAX_N = 33000                   # the largest size tested; npad 65536 (34 GB a matrix) is not


def test_schedule_table_spot_checks():
    assert [schedule(N, False) for N in (96, 97, 2048, 3000)] == \
        ["fused", "rec+levels", "rec+levels+sidesolve", "rec+rec+sidesolve"]
    assert [schedule(N, False) for N in (4096, 4097, 8192, 24577, 32768, 33000)] == \
        ["la512+levels+sidesolve", "la512+rec+sidesolve", "overlap512+sidesolve", "la1024+rec+sidesolve",
         "overlap1024+sidesolve", "la1024+rec+seqsolve"]
    assert [schedule(N, True) for N in (1921, 16384, 32768, 33000)] == \
        ["rec+levels", "overlap512", "overlap1024", "la1024+rec"]


def test_gpu_cases_reach_every_schedule():
    """Every schedule mfgp_lml_grad(_timed) and mfgp_factorize can take up to MAX_N is run by a GPU case below.
    mfgp_factorize runs the sequential solve, i.e. the timed label.  If this fails after a threshold moved in
    capi.cu / linalg.cu, update schedule() and add a size."""
    reachable = {schedule(N, t) for N in [1] + list(range(LEAF, MAX_N + LEAF, LEAF)) for t in (False, True)}
    reached = {schedule(N, False) for N in ORACLE_N + LARGE_N}
    reached |= {schedule(N, True) for N in LARGE_N}                     # factorize in the FD checks
    reached |= {schedule(N, t) for N in TIMED_N for t in (False, True)}
    reached |= {schedule(N, t) for N, _, _ in INFO_CASES for t in (False, True)}
    assert reached == reachable, sorted(reachable - reached)
    # the structured cases reach every Cholesky driver / inverse form of mfgp_potrf + mfgp_trtri below npad 32768
    assert {factor_label(n) for n in STRUCT_NPAD} == {factor_label(n) for n in range(LEAF, 32768, LEAF)}
    assert any(n >= 6144 + LEAF and n % 512 for n in STRUCT_NPAD)                # TMA row solves, ragged panel


# ---- exact structured matrices --------------------------------------------------------------------------------------
def structured_S(npad, pattern, seed=0):
    """Strictly lower S with entries in {-1, 0, 1} and S @ S = 0: the nonzero rows and the nonzero columns come
    from disjoint index sets (pattern "A": columns from the first 64 indices of every 128-tile, rows from the last
    64; "B": swapped).  Every sub-block product of S vanishes as well, so (I + S)^-1 = I - S, and every partial sum
    of the blocked Cholesky, inverse and W^T W is a small integer: exact in FP64 whatever the order.

    About 4-8 random nonzeros per row, plus one in every lower 128 x 128 tile that can hold one (the diagonal tiles
    only in pattern A) and one on the leaf edges (row = 127 / col = 0 mod 128 in A, row = 0 / col = 127 in B) of
    every tile row; so the panel edges 511/512 and 1023/1024 and, in pattern A, the last row carry nonzeros too."""
    rng = np.random.default_rng(seed + npad)
    idx = np.arange(npad)
    first = idx % LEAF < LEAF // 2
    rows_set, cols_set = (idx[~first], idx[first]) if pattern == "A" else (idx[first], idx[~first])
    r_edge, c_edge = (LEAF - 1, 0) if pattern == "A" else (0, LEAF - 1)
    R, C = [], []
    # random entries: for row i, columns drawn from the column set below i
    n_below = np.searchsorted(cols_set, rows_set)          # columns of the set with j < i
    k = rng.integers(4, 9, size=rows_set.size)
    for kk in range(8):
        sel = (kk < k) & (n_below > 0)
        R.append(rows_set[sel])
        C.append(cols_set[(rng.random(sel.sum()) * n_below[sel]).astype(np.int64)])
    # one entry per lower tile (J < I; J == I for pattern A), and on the leaf edges
    m = npad // LEAF
    I, J = np.tril_indices(m, 0 if pattern == "A" else -1)
    half = LEAF // 2
    roff = np.where(first[:LEAF])[0] if pattern == "B" else np.where(~first[:LEAF])[0]
    coff = np.where(~first[:LEAF])[0] if pattern == "B" else np.where(first[:LEAF])[0]
    R.append(I * LEAF + roff[rng.integers(0, half, I.size)])
    C.append(J * LEAF + coff[rng.integers(0, half, J.size)])
    Ie = np.arange(m) if pattern == "A" else np.arange(1, m)
    for Je in (Ie if pattern == "A" else Ie - 1, (rng.random(Ie.size) * (Ie + (pattern == "A"))).astype(np.int64)):
        R.append(Ie * LEAF + r_edge)
        C.append(Je * LEAF + c_edge)
    R, C = np.concatenate(R), np.concatenate(C)
    assert np.all(C < R)
    key = np.unique(R * npad + C)
    R, C = key // npad, key % npad
    V = rng.choice(np.array([-1, 1], dtype=np.int64), size=R.size)
    return sp.csr_matrix((V, (R, C)), shape=(npad, npad), dtype=np.int64)


def test_structured_matrices_are_nilpotent_and_cover_every_tile():
    for npad in (384, 1152):
        for pattern in ("A", "B"):
            S = structured_S(npad, pattern)
            assert (S @ S).count_nonzero() == 0
            Sd = S.toarray()
            assert np.all(np.triu(Sd) == 0) and set(np.unique(Sd)) == {-1, 0, 1}
            m = npad // LEAF
            tiles = np.abs(Sd).reshape(m, LEAF, m, LEAF).sum(axis=(1, 3)) > 0
            assert np.all(tiles[np.tril_indices(m, 0 if pattern == "A" else -1)])
            nnz = np.diff(S.indptr)
            assert np.median(nnz[nnz > 0]) >= 4
            edge_r, edge_c = (LEAF - 1, 0) if pattern == "A" else (0, LEAF - 1)
            assert np.all(np.abs(Sd[edge_r::LEAF]).sum(axis=1)[pattern == "B":] > 0)
            assert np.abs(Sd[:, edge_c::LEAF]).sum() > 0
            if npad < 1152:
                continue
            if pattern == "A":      # panel edges: rows 511 and 1023, columns 512 and 1024; the last row
                assert nnz[511] > 0 and nnz[1023] > 0 and nnz[-1] > 0
                assert np.any(Sd[:, 512]) and np.any(Sd[:, 1024])
            else:
                assert Sd[512, 511] != 0 and Sd[1024, 1023] != 0
    # the inverse of the unit factor is I - S, exactly
    S = structured_S(384, "A").toarray()
    I = np.eye(384)
    assert np.array_equal((I + S) @ (I - S), I)


# ---- GPU fixtures and helpers ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def T(gpu):
    from multifidelity_datafusion_gps_b200 import ops

    class NS:
        pass
    ns = NS()
    ns.ops, ns.dev = ops, "cuda:0"
    ns.up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to("cuda:0")
    return ns


@pytest.fixture
def room(T):
    """room(npad, k=4): skip unless k npad x npad FP64 matrices plus a margin fit in free device memory (the
    machines are shared).  Frees the case's buffers afterwards."""
    def need(npad, k=4):
        free, _ = torch.cuda.mem_get_info()
        want = k * npad * npad * 8 + (2 << 30)
        if free < want:
            pytest.skip("needs %.1f GB of free device memory, %.1f GB free" % (want / 2 ** 30, free / 2 ** 30))
    yield need
    gc.collect()
    torch.cuda.empty_cache()


def _dense(T, S, npad):
    """Sparse integer matrix -> dense FP64 device matrix (built on the device, exact)."""
    C = S.tocoo()
    out = torch.zeros((npad, npad), dtype=torch.float64, device=T.dev)
    r = torch.from_numpy(C.row.astype(np.int64)).to(T.dev)
    c = torch.from_numpy(C.col.astype(np.int64)).to(T.dev)
    out.index_put_((r, c), torch.from_numpy(C.data.astype(np.float64)).to(T.dev))
    return out


BLOCK = 4096


def _tril_rows(M, r0, r1, n):
    return torch.tril(M[r0:r1, :n], diagonal=r0)


def _tril_mm(M, B, n):
    """tril(M)[:n, :n] @ B, a row block at a time (no n x n copy)."""
    out = torch.empty((n, B.shape[1]), dtype=B.dtype, device=B.device)
    for r0 in range(0, n, BLOCK):
        r1 = min(n, r0 + BLOCK)
        out[r0:r1] = _tril_rows(M, r0, r1, n) @ B
    return out


def _sym_mm(M, B, n):
    """(tril(M) + tril(M, -1)^T)[:n, :n] @ B, the symmetric matrix stored in M's lower triangle."""
    out = torch.zeros((n, B.shape[1]), dtype=B.dtype, device=B.device)
    for r0 in range(0, n, BLOCK):
        r1 = min(n, r0 + BLOCK)
        Mb = _tril_rows(M, r0, r1, n)
        out[r0:r1] += Mb @ B
        out += Mb.T @ B[r0:r1]
    return out - M.diagonal()[:n, None] * B


def _tril_equal(X, Y, n):
    return all(torch.equal(_tril_rows(X, r0, min(n, r0 + BLOCK), n), _tril_rows(Y, r0, min(n, r0 + BLOCK), n))
               for r0 in range(0, n, BLOCK))


# ---- 1. exact arithmetic: potrf, trtri, lauum bit for bit -----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["A", "B"])
@pytest.mark.parametrize("npad", STRUCT_NPAD)
def test_structured_factor_inverse_and_kinv_are_exact(T, room, npad, pattern):
    """A = (I + S)(I + S)^T with S from structured_S: potrf(A) = I + S, trtri = I - S and the lower triangle of
    lauum = that of (I - S)^T (I - S), compared with torch.equal.  Every product and sum is of small integers, so
    any tile mask, batch stride or panel edge error shows as a wrong integer, never as rounding.  This relies on
    the leaf kernel's rsqrt(1.0) being exactly 1.0 (linalg.cu:52), as it is on sm_100a; npad = 128 would be the
    first case to show otherwise."""
    room(npad, 5)
    S = structured_S(npad, pattern)
    I = sp.identity(npad, dtype=np.int64, format="csr")
    Ap = _dense(T, (I + S) @ (I + S).T, npad)
    W, info = T.ops.potrf(Ap)
    assert info == 0
    L0 = _dense(T, I + S, npad)
    L = torch.tril(Ap)
    del Ap
    if not torch.equal(L, L0):
        bad = (L != L0).nonzero()
        pytest.fail("potrf: %d wrong entries, first at %s, max |err| %.3g" %
                    (bad.shape[0], bad[0].tolist(), (L - L0).abs().max().item()))
    del L0
    T.ops.trtri(L, W)
    Winv = torch.tril(W)
    ref = _dense(T, I - S, npad)
    if not torch.equal(Winv, ref):
        bad = (Winv != ref).nonzero()
        pytest.fail("trtri: %d wrong entries, first at %s" % (bad.shape[0], bad[0].tolist()))
    del L, Winv, ref
    Kinv = torch.tril(T.ops.lauum(W))
    del W
    ref = torch.tril(_dense(T, (I - S).T @ (I - S), npad))
    if not torch.equal(Kinv, ref):
        bad = (Kinv != ref).nonzero()
        pytest.fail("lauum: %d wrong entries, first at %s" % (bad.shape[0], bad[0].tolist()))


# ---- 2. random GP covariances ---------------------------------------------------------------------------------------
def _case(N):
    return util.random_case(100 + N, N, d, E, KIND)


@pytest.mark.gpu
@pytest.mark.parametrize("N", ORACLE_N)
def test_lml_grad_matches_oracle_at_schedule_boundaries(T, room, N):
    """Side-stream solves (npad 2048, 3072), look-ahead Cholesky with the batched inverse (4095) and with the
    recursive one on a ragged last panel (4097), against the NumPy oracle with the bounds of
    test_lml_and_gradient_match_oracle."""
    room(padded(N), 3)
    X, Y, th = _case(N)
    buf = T.ops.FactorBuffers(N, T.dev)
    lml, g, info = T.ops.lml_grad(T.up(X), T.up(Y.ravel()), KIND, d, th, buf)
    assert info == 0
    alpha = buf.alpha.cpu().numpy()[:N]
    Ki = np.tril(buf.A[:N, :N].cpu().numpy())
    del buf
    for form, tol in (("direct", 1e-9), ("gpy", 1e-6)):
        ref = go.inference(KIND, X, Y, d, th, form=form)
        errs = (abs(lml - ref["lml"]) / abs(ref["lml"]), util.rel_err(g, ref["grad"]),
                util.rel_err(alpha, ref["alpha"].ravel()), util.rel_err(Ki, np.tril(ref["Ki"])))
        print("N=%d %s: lml %.2e grad %.2e alpha %.2e Ki %.2e" % ((N, form) + errs))
        assert errs[0] <= tol
        assert errs[1] < max(tol, 1e-8)
        assert errs[2] < max(tol, 1e-8)
        assert errs[3] < max(tol, 1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("N", LARGE_N)
def test_large_fit_against_cusolver_and_properties(T, room, N):
    """Sizes where the O(N^3) oracle is too slow: look-ahead with the recursive inverse (10000), 1024-wide panels
    (24577), their overlapped form (32768) and the sequential solve beyond the side stream's scratch (33000).
    L against torch.linalg.cholesky (cuSOLVER, the checker only) element by element, the LML recomputed from that
    factor, L L^T = K_y, W L = I and K^-1 K_y = I on sampled columns, K_y alpha = y, and two gradient entries
    against central differences of the GPU LML."""
    npad = padded(N)
    room(npad, 4)
    X, Y, th = _case(N)
    dX, dy = T.up(X), T.up(Y.ravel())
    buf = T.ops.FactorBuffers(N, T.dev)
    lml, logdet, yta, info = T.ops.factorize(dX, dy, KIND, d, th, buf)
    assert info == 0 and np.isfinite(lml)
    Ky = T.ops.assemble(dX, KIND, d, th, uplo=1)
    cols = torch.arange(5, N, N // 16, device=T.dev)
    Ky_cols = Ky[:, cols].clone()
    res_alpha = ((Ky @ buf.alpha[:N] - dy).abs().max() / dy.abs().max()).item()
    Lref = torch.linalg.cholesky(Ky)
    del Ky
    scale = Lref.abs().max().item()
    err_L = max((_tril_rows(buf.A, r0, min(N, r0 + BLOCK), N) - Lref[r0:r0 + BLOCK]).abs().max().item()
                for r0 in range(0, N, BLOCK)) / scale
    ld_ref = 2.0 * torch.log(Lref.diagonal()).sum().item()
    v = torch.linalg.solve_triangular(Lref, dy[:, None], upper=False)
    lml_ref = 0.5 * (-N * np.log(2 * np.pi) - ld_ref - (v * v).sum().item())
    del Lref, v
    n_c = cols.numel()
    E_cols = torch.zeros((N, n_c), dtype=torch.float64, device=T.dev)
    E_cols[cols, torch.arange(n_c, device=T.dev)] = 1.0
    ar = torch.arange(N, device=T.dev)
    Lc_rows = torch.where(ar[None, :] <= cols[:, None], buf.A[cols, :N], 0.0)     # rows `cols` of L
    Lc_cols = torch.where(ar[:, None] >= cols[None, :], buf.A[:N, cols], 0.0)     # columns `cols` of L
    err_LLt = (_tril_mm(buf.A, Lc_rows.T, N) - Ky_cols).abs().max().item()
    err_WL = (_tril_mm(buf.W, Lc_cols, N) - E_cols).abs().max().item()
    alpha = buf.alpha[:N].clone()
    lml2, g, info = T.ops.lml_grad(dX, dy, KIND, d, th, buf)
    assert info == 0
    err_KiK = (_sym_mm(buf.A, Ky_cols, N) - E_cols).abs().max().item()
    err_Kiy = ((_sym_mm(buf.A, dy[:, None], N).ravel() - alpha).abs().max() / alpha.abs().max()).item()
    fd_err = []
    for i in (1, 6):
        hstep = 1e-5 * th[i]
        tp, tm = th.copy(), th.copy()
        tp[i] += hstep
        tm[i] -= hstep
        fd = (T.ops.factorize(dX, dy, KIND, d, tp, buf)[0] - T.ops.factorize(dX, dy, KIND, d, tm, buf)[0]) / (2 * hstep)
        fd_err.append(abs(g[i] - fd) / max(1.0, abs(fd)))
    print("N=%d: L-vs-cusolver %.2e lml-vs-cusolver %.2e (lml2 %.2e) LLt %.2e WL %.2e KiK %.2e Kiy %.2e "
          "Ky.alpha %.2e fd %s" % (N, err_L, abs(lml - lml_ref) / abs(lml_ref), abs(lml2 - lml) / abs(lml), err_LLt,
                                  err_WL, err_KiK, err_Kiy, res_alpha, fd_err))
    # bounds ~30x above what an NVIDIA B200 (1000 W limit) gives on these seeded cases: L against cuSOLVER <= 2.2e-13,
    # LML 2.0e-13, L L^T 1.6e-14, W L 7.6e-14, K^-1 K_y 3.3e-12, K^-1 y 7.7e-14, K_y alpha 7.1e-12; the central
    # differences' own truncation error (up to 2.2e-7) sets the gradient bound of test_full_size_lml_grad_properties
    assert err_L < 1e-11
    assert abs(lml - lml_ref) <= 1e-11 * abs(lml_ref)
    assert abs(lml2 - lml) <= 1e-12 * abs(lml)
    assert err_LLt < 1e-12
    assert err_WL < 1e-11
    assert err_KiK < 1e-10
    assert err_Kiy < 1e-11
    assert res_alpha < 1e-10
    assert max(fd_err) <= 2e-5


# ---- 3. timed against untimed schedule ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N", TIMED_N)
def test_timed_and_untimed_schedules_agree_bit_for_bit(T, room, N):
    """mfgp_lml_grad_timed with stage events runs the solves after K^-1 = W^T W on one stream; without, from
    npad 2048 to 32768, they run on the side stream under it.  Both launch the same kernels on the same data, so
    the LML, the gradient, alpha, K^-1 and W must agree bit for bit, and so must two untimed calls."""
    npad = padded(N)
    room(npad, 4)
    X, Y, th = _case(N)
    dX, dy = T.up(X), T.up(Y.ravel())
    buf = T.ops.FactorBuffers(N, T.dev)
    lml_u, g_u, info = T.ops.lml_grad(dX, dy, KIND, d, th, buf)
    assert info == 0
    A_u, W_u, al_u = buf.A.clone(), buf.W.clone(), buf.alpha[:N].clone()

    def same():
        return (torch.equal(buf.alpha[:N], al_u), _tril_equal(buf.A, A_u, N), _tril_equal(buf.W, W_u, N))

    lml_t, g_t, info, ms = T.ops.lml_grad(dX, dy, KIND, d, th, buf, timed=True)
    assert info == 0 and np.all(ms >= 0)
    assert lml_t == lml_u and np.array_equal(g_t, g_u)
    assert same() == (True, True, True), "timed against untimed: alpha, K^-1, W"
    lml_2, g_2, info = T.ops.lml_grad(dX, dy, KIND, d, th, buf)
    assert info == 0 and lml_2 == lml_u and np.array_equal(g_2, g_u)
    assert same() == (True, True, True), "two untimed calls: alpha, K^-1, W"


# ---- 4. first bad pivot ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N,rows,expected", INFO_CASES)
def test_first_bad_pivot_in_every_schedule(T, room, N, rows, expected):
    """A NaN in row r of X makes pivot r the first that is not positive: mfgp_factorize and mfgp_lml_grad return
    r + 1 (with two NaN rows, the lower index).  A good call on the same handle afterwards returns 0."""
    room(padded(N), 3)
    X, Y, th = _case(N)
    Xbad = X.copy()
    Xbad[rows] = np.nan
    dy = T.up(Y.ravel())
    buf = T.ops.FactorBuffers(N, T.dev)
    assert T.ops.factorize(T.up(Xbad), dy, KIND, d, th, buf)[3] == expected
    assert T.ops.lml_grad(T.up(Xbad), dy, KIND, d, th, buf)[2] == expected
    assert T.ops.factorize(T.up(X), dy, KIND, d, th, buf)[3] == 0
    assert T.ops.lml_grad(T.up(Xbad), dy, KIND, d, th, buf)[2] == expected
    assert T.ops.lml_grad(T.up(X), dy, KIND, d, th, buf)[2] == 0


@pytest.mark.gpu
def test_potrf_reports_negative_pivot_on_lookahead_path(T, room):
    npad, k = 6272, 5555
    room(npad, 3)
    A = torch.eye(npad, dtype=torch.float64, device=T.dev)
    A[k, k] = -1.0
    _, info = T.ops.potrf(A)
    assert info == k + 1
    A = torch.eye(npad, dtype=torch.float64, device=T.dev)
    _, info = T.ops.potrf(A)
    assert info == 0
