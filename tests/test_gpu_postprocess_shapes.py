"""The device kernels that run after the trace — dense AP / DkAP smoothing, sparse AP, the grey GMRES solve and the CSR / CSC
read-out of the resident counts — at the shapes where their hard-coded boundaries sit: rows padded to 16 doubles, 32 x 32
tiles, 1024-thread row loops that wrap only past 1024 / 2048 elements, the single-block scan, 64-row CSC tiles, warp-per-row
sparse kernels, the radix-sort key width changing at 2^16, the matvec row tiles and unroll tails, and the 32 MB pieces of a
pageable copy.

Every reference here is written independently of the library, in numpy longdouble (80-bit on x86) or exact integers:
  * dense / sparse AP are compared iteration for iteration (max_iters 0..3) at ~1e-13 relative, and the reported
    delta_init / delta against delta_R_X at 1e-12 relative plus the rounding slack of u_i - u_j — a single wrong scaling
    pass cannot be washed out by later iterations, as it can after convergence;
  * the solve is checked through g = F'j and the residual recomputed from the returned j, whether or not GMRES converged;
  * the count read-outs are compared bit for bit with host integers (CSC divides by the row total, CSR multiplies by its
    reciprocal — both exactly reproducible in float64).
The tests without the `gpu` mark check the references themselves against smoothing.AP / DkAP and numpy.linalg.solve, so a
broken reference cannot make a device test pass."""
import numpy as np
import pytest
import scipy.sparse as sp

LD = np.longdouble
EPS = np.finfo(np.float64).eps
TARGET = 8 * EPS


# ------------------------------------------------------------------------------------------------------------------------------
# references (longdouble / exact integers)
# ------------------------------------------------------------------------------------------------------------------------------
def _delta_terms(Xp, ui, uj, wi, wj):
    """delta_R_X over the pairs given (i < j) and the rounding slack of a float64 evaluation: u_i - u_j cancels, so an
    error of 64 eps |u| in u shifts every term by up to 2 |X_ij|^2 |u_i - u_j| 64 eps (|u_i| + |u_j|) / (w_i^2 + w_j^2).
    Returns (delta, slack on delta)."""
    du = ui - uj
    den = wi ** 2 + wj ** 2
    d2 = ((Xp * du) ** 2 / den).sum()
    e2 = (2 * Xp ** 2 * np.abs(du) * 64 * LD(EPS) * (np.abs(ui) + np.abs(uj)) / den).sum()
    delta = np.sqrt(d2)
    return delta, (e2 / (2 * delta) if delta > 0 else LD(0))


def _delta_dense(X, u, w):
    """delta_R_X: sqrt(sum_{i<j} (X_ij (u_i - u_j))^2 / (w_i^2 + w_j^2)), and its float64 rounding slack."""
    i, j = np.triu_indices(len(u), 1)
    return _delta_terms(X[i, j], u[i], u[j], w[i], w[j])


def ref_ap_dense(F, w, iters):
    """AP restated in longdouble on a dense F: X = (WF + (WF)')/2, `iters` scalings X_ij *= (u_i + u_j)/2 with u = w ./ r
    (u = 1 on an empty row), F = X ./ r.  Returns [(F_k, (delta_k, slack_k)) for k = 0..iters]."""
    F = np.asarray(F, dtype=LD)
    w = np.asarray(w, dtype=LD)
    WF = w[:, None] * F
    X = (WF + WF.T) / 2
    out = []
    for k in range(iters + 1):
        if k:
            X = X * ((u[:, None] + u[None, :]) / 2)
        r = X.sum(axis=1)
        pos = r > 0
        u = np.where(pos, w / np.where(pos, r, 1), LD(1))
        out.append((X / np.where(pos, r, 1)[:, None] * pos[:, None], _delta_dense(X, u, w)))
    return out


def ref_F_from_counts(c):
    """F = counts / row total, exact integers in longdouble (u64 < 2^64 fits the 64-bit mantissa)."""
    cl = np.asarray(c).astype(LD)
    rs = cl.sum(axis=1, keepdims=True)
    return np.where(rs > 0, cl / np.where(rs > 0, rs, 1), LD(0))


def union_pattern(F):
    """Pattern of WF + (WF)' (all values positive: no cancellation), CSR with sorted columns."""
    A = sp.csr_matrix(F, dtype=np.float64, copy=True)
    A.data = np.ones_like(A.data)
    P = (A + A.T).tocsr()
    P.sort_indices()
    return P.indptr.astype(np.int64), P.indices.astype(np.int64)


def _lookup(F, rows, cols):
    """F[rows, cols] (0 where F has no entry), vectorised over a sorted key table."""
    C = sp.coo_matrix(F)
    n = F.shape[0]
    keys = C.row.astype(np.int64) * n + C.col.astype(np.int64)
    order = np.argsort(keys)
    keys, vals = keys[order], C.data[order]
    q = rows * n + cols
    pos = np.searchsorted(keys, q)
    pos_c = np.minimum(pos, max(len(keys) - 1, 0))
    hit = (pos < len(keys)) & (keys[pos_c] == q) if len(keys) else np.zeros(len(q), bool)
    return np.where(hit, vals[pos_c] if len(keys) else 0.0, 0.0)


def ref_ap_sparse(F, w, iters):
    """AP restated in longdouble on the union pattern (CSR of X).  Returns (indptr, cols, [(vals_k, delta_k)]) with vals_k
    the entries of F_smooth_k in the CSR order of the pattern (row i, column j)."""
    n = F.shape[0]
    indptr, cols = union_pattern(F)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(indptr))
    w = np.asarray(w, dtype=LD)
    fij = _lookup(F, rows, cols).astype(LD)
    fji = _lookup(F, cols, rows).astype(LD)
    X = (w[rows] * fij + w[cols] * fji) / 2
    empty = np.diff(indptr) == 0
    upper = cols > rows
    out = []
    for k in range(iters + 1):
        if k:
            X = X * ((u[rows] + u[cols]) / 2)
        r = np.add.reduceat(np.append(X, LD(0)), np.minimum(indptr[:-1], len(X))) if n else X[:0]
        r[empty] = 0
        pos = r > 0
        u = np.where(pos, w / np.where(pos, r, 1), LD(1))
        ru, cu = rows[upper], cols[upper]
        rr = np.where(pos, r, 1)[rows]
        out.append((np.where(pos[rows], X / rr, LD(0)), _delta_terms(X[upper], u[ru], u[cu], w[ru], w[cu])))
    return indptr, cols, out


def _csr_order_to_csc(indptr, cols, n):
    """Permutation from the CSR order (row, col) of a pattern to the CSC order (col, row) of the same entries."""
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(indptr))
    return np.lexsort((rows, cols))


def ref_matvec_t(F, x):
    """F'x in longdouble for dense or sparse F."""
    if sp.issparse(F):
        C = sp.coo_matrix(F)
        y = np.zeros(F.shape[1], dtype=LD)
        np.add.at(y, C.col, C.data.astype(LD) * np.asarray(x, dtype=LD)[C.row])
        return y
    return np.asarray(F, dtype=LD).T @ np.asarray(x, dtype=LD)


def _abs(F):
    return abs(F) if sp.issparse(F) else np.abs(F)


def _max_rel(got, ref):
    ref = np.asarray(ref, dtype=LD)
    d = np.abs(np.asarray(got, dtype=LD) - ref)
    nz = ref != 0
    if np.any(d[~nz] != 0):
        return np.inf
    return float((d[nz] / np.abs(ref[nz])).max()) if nz.any() else 0.0


def _delta_ok(got, ref):
    """Reported delta against (delta, slack) of the reference: 1e-12 relative plus the cancellation slack of u_i - u_j."""
    d, slack = ref
    return abs(LD(got) - d) <= LD(1e-12) * d + slack if d != 0 else got == 0.0


# ------------------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------------------
def dense_F(n, seed, zero=False):
    """Positive F with unit row sums, some all-zero rows and some zero columns whose rows are not zero."""
    rng = np.random.default_rng(seed)
    F = rng.random((n, n)) + 1e-3
    if zero:
        return np.zeros((n, n))
    if n >= 3:
        idx = rng.permutation(n)
        k = max(1, n // 64)
        F[idx[:k], :] = 0.0                              # empty rows
        F[:, idx[k:2 * k]] = 0.0                         # empty columns, their rows are not empty
    rs = F.sum(axis=1, keepdims=True)
    return np.divide(F, rs, out=np.zeros_like(F), where=rs > 0)


def dense_counts(n, seed, zero=False):
    """u64 counts with entries above 2^32, one row total above 2^53 (all below 2^60), zero entries, an empty row and an
    empty column."""
    rng = np.random.default_rng(seed)
    if zero:
        return np.zeros((n, n), np.uint64)
    top = 59 - int(np.ceil(np.log2(max(n, 2))))        # n * 2^top <= 2^59
    bits = rng.integers(20, top + 1, n)
    bits[0] = top
    c = np.empty((n, n), np.uint64)
    for i in range(n):
        c[i] = rng.integers(0, np.uint64(1) << np.uint64(bits[i]), n, dtype=np.uint64)
    c[rng.random((n, n)) < 0.2] = 0
    c[0, 0] = np.uint64(1) << np.uint64(top)
    if n >= 3:
        c[n // 2, :] = 0
        c[:, n // 3] = 0
        c[n // 3, 0] = 5
    return c


def weights(n, seed):
    return np.random.default_rng(seed + 7).uniform(1.0, 10.0, n)


def sparse_random(n, per_row, seed):
    """~per_row entries per row at random positions (some rows and columns empty), positive values, unit row sums."""
    rng = np.random.default_rng(seed)
    m = n * per_row
    A = sp.coo_matrix((rng.random(m) + 1e-3, (rng.integers(0, n, m), rng.integers(0, n, m))), shape=(n, n)).tocsr()
    A.sum_duplicates()
    rs = np.asarray(A.sum(axis=1)).ravel()
    A = sp.diags(np.divide(1.0, rs, out=np.zeros(n), where=rs > 0)) @ A
    return A.tocsc()


def sparse_structured(seed):
    """n = 200: row 0 full, column 1 full but for the empty row 7 (whose column is not empty), X rows of exactly 31, 32, 33, 64
    and 65 entries, F_ij != 0 with F_ji = 0, and diagonal entries."""
    rng = np.random.default_rng(seed)
    n = 200
    F = np.zeros((n, n))
    special = {2: 31, 3: 32, 4: 33, 5: 64, 6: 65}
    free = np.setdiff1d(np.arange(8, n), list(special))
    for i in range(8, n):                                  # upper-triangle entries only: F_ij != 0, F_ji == 0
        cand = free[free > i]
        if len(cand):
            F[i, rng.choice(cand, min(3, len(cand)), replace=False)] = rng.random(min(3, len(cand))) + 0.1
        if i % 3 == 0:
            F[i, i] = rng.random() + 0.1                   # diagonal
    F[:, 1] = rng.random(n) + 0.1                          # full column
    F[0, :] = rng.random(n) + 0.1                          # full row
    for i, L in special.items():                           # X row i = F row i exactly: nobody else points at i except row 0
        cols = np.concatenate(([0, 1], rng.choice(free, L - 2, replace=False)))
        F[i, :] = 0.0
        F[i, cols] = rng.random(L) + 0.1
    F[8, 7] = 0.5                                          # row 7 empty, column 7 not
    F[0, 7] = 0.25
    F[7, :] = 0.0
    Fx = sp.csc_matrix(F)
    X_len = np.diff(union_pattern(Fx)[0])
    assert [X_len[i] for i in special] == list(special.values())
    assert np.diff(Fx.indptr)[1] == n - 1 and (F[0] > 0).all() and not F[7].any() and F[:, 7].any()
    return Fx


def grey_system(n, seed, kind):
    """F (dense, or CSC with empty rows and columns), coeff in [0, 0.6], rhs."""
    rng = np.random.default_rng(seed)
    if kind == "csc":
        F = sparse_random(n, 4, seed).toarray()
        if n >= 4:
            F[n // 3, :] = 0.0
            F[:, n // 2] = 0.0
        F = sp.csc_matrix(F)
    else:
        F = rng.random((n, n))
        F /= F.sum(axis=1, keepdims=True)
    coeff = rng.uniform(0.0, 0.6, n)
    h = rng.random(n) * 1e3
    return F, coeff, h


def num_elements_of(a, b):
    return 2 * a + 2 * b + a * b


NDIV = {62: (4, 9), 64: (2, 15), 128: (2, 31), 1023: (11, 77), 1024: (2, 255), 1025: (19, 47), 2047: (5, 291),
        2048: (2, 511)}


# ------------------------------------------------------------------------------------------------------------------------------
# 6. the references themselves (no GPU)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 17, 40])
def test_dense_reference_reproduces_numpy_ap(rthx_mod, n):
    F = dense_F(n, 11 + n)
    w = weights(n, n)
    snaps = ref_ap_dense(F, w, 3)
    for k, (Fk, _) in enumerate(snaps):
        got = rthx_mod.smoothing.AP(F, w, max(n - 1, 0), max_iters=k)
        assert _max_rel(got, Fk) < 1e-13
    assert snaps[0][1][0] > 0 or n == 1
    # delta_R_X is a plain sum over the upper triangle
    X = (w[:, None] * F + (w[:, None] * F).T) / 2
    r = X.sum(axis=1)
    u = np.where(r > 0, w / np.where(r > 0, r, 1), 1.0)
    d2 = sum((X[i, j] * (u[i] - u[j])) ** 2 / (w[i] ** 2 + w[j] ** 2) for i in range(n) for j in range(i + 1, n))
    assert abs(float(snaps[0][1][0]) - np.sqrt(d2)) <= 1e-12 * max(np.sqrt(d2), 1e-300)


def test_dense_reference_from_counts_and_dkap(rthx_mod):
    c = dense_counts(20, 3)
    F = ref_F_from_counts(c)
    rs = c.astype(object).sum(axis=1)                                  # exact Python integers
    assert max(rs) > 2 ** 53 and max(rs) < 2 ** 60 and c.max() > 2 ** 32
    assert (c[10] == 0).all() and (c[:, 6] == 0).all() and c[6].any()
    for i in (0, 1, 5):
        assert abs(float(F[i, 3]) - float(c[i, 3]) / float(rs[i])) <= 2 * EPS * float(F[i, 3])
    w = weights(20, 3)
    Fd = dense_F(20, 5)
    Fd[Fd.sum(axis=1) == 0, 0] = 1.0                                   # DkAP needs non-empty rows
    ref = ref_ap_dense(Fd, w, 2)
    assert _max_rel(rthx_mod.smoothing.DkAP(Fd, w, 5, k_dykstra=0, max_iters=2), ref[2][0]) < 1e-13


@pytest.mark.parametrize("case", ["structured", "random", "one_entry", "empty"])
def test_sparse_reference_reproduces_numpy_ap(rthx_mod, case):
    if case == "structured":
        F = sparse_structured(1)
    elif case == "random":
        F = sparse_random(300, 8, 2)
    elif case == "one_entry":
        F = sp.csc_matrix(np.array([[0.7]]))
    else:
        F = sp.csc_matrix((50, 50))
    n = F.shape[0]
    w = weights(n, 4)
    indptr, cols, snaps = ref_ap_sparse(F, w, 3)
    dense = ref_ap_dense(F.toarray(), w, 3)
    for k, (vals, delta) in enumerate(snaps):
        got = rthx_mod.smoothing.AP(F, w, max(n - 1, 0), max_iters=k).tocsr()
        got.sort_indices()
        assert np.array_equal(got.indptr, indptr) and np.array_equal(got.indices, cols)
        assert _max_rel(got.data, vals) < 1e-13
        rows = np.repeat(np.arange(n), np.diff(indptr))
        assert _max_rel(np.asarray(dense[k][0][rows, cols], np.float64), vals) < 1e-13
        assert abs(delta[0] - dense[k][1][0]) <= 1e-15 * abs(dense[k][1][0])


def test_solve_reference_and_ndiv_table(rthx_mod):
    for kind in ("dense", "csc"):
        F, coeff, h = grey_system(60, 9, kind)
        Fd = F.toarray() if sp.issparse(F) else F
        j = np.linalg.solve(np.eye(60) - coeff[:, None] * Fd.T, h)
        g = ref_matvec_t(F, j)
        assert _max_rel(Fd.T @ j, g) < 1e-12
        res = np.sqrt(np.sum((h - (j - coeff * g)) ** 2))
        assert res < 1e-10 * np.linalg.norm(h)
    if kind == "csc":
        assert (np.diff(F.indptr) == 0).any() and (np.asarray(F.sum(axis=1)).ravel() == 0).any()
    for N, (a, b) in NDIV.items():
        assert num_elements_of(a, b) == N
        assert rthx_mod.meshes.square_domain(Ndiv=(a, b)).num_elements == N


# ------------------------------------------------------------------------------------------------------------------------------
# 1. dense AP and DkAP
# ------------------------------------------------------------------------------------------------------------------------------
DENSE_N = [1, 2, 15, 16, 17, 31, 32, 33, 1023, 1024, 1025, 2047, 2048, 2049]


@pytest.fixture(scope="module")
def tracer(rthx_mod, cuda_lib):
    tr = rthx_mod.DeviceTracer(rthx_mod.flatten_domain(rthx_mod.meshes.square_domain(3)), device=0)
    yield tr
    tr.close()


def _dense_case(n, source, zero=False):
    w = weights(n, n)
    if source == "F":
        src = dense_F(n, 100 + n, zero)
        return w, dict(F=src), src
    src = dense_counts(n, 200 + n, zero)
    return w, dict(counts=src), ref_F_from_counts(src)


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["F", "counts"])
@pytest.mark.parametrize("n", DENSE_N)
def test_dense_ap_iteration_matched(tracer, n, source):
    w, kw, F_ref = _dense_case(n, source)
    snaps = ref_ap_dense(F_ref, w, 3)
    for k in range(4):
        Fs, st = tracer.smooth(w, max_iters=k, **kw)
        it = st["iterations"]
        assert it == (0 if snaps[0][1][0] <= TARGET else k), (k, st)
        assert _max_rel(Fs, snaps[it][0]) < 1e-13, k
        assert _delta_ok(st["delta_init"], snaps[0][1]), (st["delta_init"], snaps[0][1])
        assert _delta_ok(st["delta"], snaps[it][1]), (k, st["delta"], snaps[it][1])


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["F", "counts"])
@pytest.mark.parametrize("n", [1, 33, 1025])
def test_dense_ap_all_zero_input(tracer, n, source):
    w, kw, _ = _dense_case(n, source, zero=True)
    Fs, st = tracer.smooth(w, max_iters=3, **kw)
    assert st["iterations"] == 0 and st["delta_init"] == 0.0 and st["delta"] == 0.0
    assert not Fs.any()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1025, 2049])
def test_dense_ap_to_convergence(rthx_mod, tracer, n):
    w, kw, F = _dense_case(n, "F")
    Fs, st = tracer.smooth(w, **kw)
    assert st["converged"] == 1 and 0 < st["iterations"] < 1000 and st["delta"] <= st["delta_init"]
    ref = rthx_mod.smoothing.AP(F, w, n - 1, max_iters=st["iterations"])
    assert np.abs(Fs - ref).max() < 1e-10
    assert np.abs(Fs.sum(axis=1) - 1.0).max() <= 1e-12
    WF = w[:, None] * Fs
    assert np.abs(WF - WF.T).max() <= 1e-12 * np.abs(WF).max()
    assert Fs.min() >= 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("k_dykstra", [1, 2, 5, 6])
@pytest.mark.parametrize("n", [17, 1025, 2049])
def test_dense_dkap_matches_numpy(rthx_mod, tracer, n, k_dykstra):
    w = weights(n, n)
    F = dense_F(n, 300 + n)
    empty = F.sum(axis=1) == 0
    F[empty, (np.flatnonzero(empty) + 1) % n] = 1.0         # numpy DkAP renormalises rows: no empty rows
    ref = rthx_mod.smoothing.DkAP(F, w, n // 2, k_dykstra=k_dykstra, max_iters=0)
    Fs, st = tracer.smooth(w, F=F, k_dykstra=k_dykstra, max_iters=0)
    assert st["iterations"] == 0 and st["dykstra_rounds"] == k_dykstra and np.isfinite(st["dykstra_delta"])
    assert np.abs(Fs - ref).max() < 1e-10
    c = dense_counts(n, 400 + n)
    c[c.sum(axis=1) == 0, 0] = 3
    Fc = (c.astype(np.float64) / c.sum(axis=1, keepdims=True).astype(np.float64))
    ref_c = rthx_mod.smoothing.DkAP(Fc, w, n // 2, k_dykstra=k_dykstra, max_iters=0)
    Fs_c, st_c = tracer.smooth(w, counts=c, k_dykstra=k_dykstra, max_iters=0)
    assert st_c["dykstra_rounds"] == k_dykstra and np.abs(Fs_c - ref_c).max() < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("n", [400, 2049])
def test_dense_pageable_out_equals_pinned(tracer, n):
    """out= with a plain (pageable) array takes the staged 2-D copy: 1.28 MB in one piece, 33.6 MB in two 32 MB pieces."""
    w, kw, _ = _dense_case(n, "F")
    F_pinned, st = tracer.smooth(w, max_iters=5, **kw)
    F_pinned = F_pinned.copy()
    out = np.full((n, n), np.nan)
    F_page, st2 = tracer.smooth(w, max_iters=5, out=out, **kw)
    assert F_page is out or np.shares_memory(F_page, out)
    assert np.array_equal(out, F_pinned) and st["delta"] == st2["delta"]


# ------------------------------------------------------------------------------------------------------------------------------
# 2. sparse AP
# ------------------------------------------------------------------------------------------------------------------------------
SPARSE_CASES = ["n1_one", "n1_empty", "all_empty", "structured", 1025, 2049, 65535, 65536, 65537, 70001]


def _sparse_case(case):
    if case == "n1_one":
        return sp.csc_matrix(np.array([[0.3]]))
    if case == "n1_empty":
        return sp.csc_matrix((1, 1))
    if case == "all_empty":
        return sp.csc_matrix((300, 300))
    if case == "structured":
        return sparse_structured(7)
    return sparse_random(case, 8, case)


def _check_sparse(Fs, st, indptr, cols, snaps, k):
    n = len(indptr) - 1
    perm = _csr_order_to_csc(indptr, cols, n)
    # X is symmetric, so the CSC of F_smooth has the pattern's row pointers as column pointers
    assert np.array_equal(Fs.indptr.astype(np.int64), indptr)
    assert np.array_equal(Fs.indices.astype(np.int64), np.repeat(np.arange(n), np.diff(indptr))[perm])
    it = st["iterations"]
    assert it == (0 if snaps[0][1][0] <= TARGET else k), (k, st)
    assert _max_rel(Fs.data, snaps[it][0][perm]) < 1e-13
    assert _delta_ok(st["delta_init"], snaps[0][1]) and _delta_ok(st["delta"], snaps[it][1])


@pytest.mark.gpu
@pytest.mark.parametrize("case", SPARSE_CASES)
def test_sparse_ap_iteration_matched(tracer, case):
    F = _sparse_case(case)
    n = F.shape[0]
    w = weights(n, 17)
    indptr, cols, snaps = ref_ap_sparse(F, w, 3)
    for k in range(4):
        Fs, st = tracer.smooth_sparse(w, F=F, max_iters=k)
        _check_sparse(Fs, st, indptr, cols, snaps, k)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["structured", 70001])
def test_sparse_ap_to_convergence(rthx_mod, tracer, case):
    F = _sparse_case(case)
    n = F.shape[0]
    w = weights(n, 19)
    Fs, st = tracer.smooth_sparse(w, F=F, max_iters=300)
    ref = rthx_mod.smoothing.AP(F, w, n - 1, max_iters=st["iterations"])
    ref.sort_indices()
    assert np.array_equal(Fs.indptr, ref.indptr) and np.array_equal(Fs.indices, ref.indices)
    assert np.abs(Fs.data - ref.data).max() < 1e-10
    assert Fs.data.min() >= 0.0 and st["delta"] <= st["delta_init"]


@pytest.mark.gpu
def test_sparse_resident_crop_is_bit_identical_to_host_csc(rthx_mod, cuda_lib):
    """From the resident counts cropped to n (row totals over the crop) == FROM_CSC on the host-cropped F built as
    float64(count) / float64(crop row total)."""
    rtm = rthx_mod.meshes.square_domain(9, kappa=3.0)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    N, ns = flat.n_elements, flat.n_surfaces
    counts = tr.trace(300, seed=81)["counts"][0].copy()
    w = weights(N, 81)
    for n in (64, 65, ns, ns + 1, N - 1):
        c = counts[:n, :n]
        rs = c.sum(axis=1)
        Fd = np.zeros((n, n))
        nz = c != 0
        Fd[nz] = c[nz].astype(np.float64) / np.repeat(rs.astype(np.float64), nz.sum(axis=1))
        Fh = sp.csc_matrix(Fd)
        for it in (2, 1000):
            Fa, sa = tr.smooth_sparse(w[:n], n=n, max_iters=it)
            Fa = sp.csc_matrix((Fa.data.copy(), Fa.indices.copy(), Fa.indptr.copy()), shape=Fa.shape)
            Fb, sb = tr.smooth_sparse(w[:n], n=n, F=Fh, max_iters=it)
            assert np.array_equal(Fa.indptr, Fb.indptr) and np.array_equal(Fa.indices, Fb.indices)
            assert np.array_equal(Fa.data, Fb.data), n
            assert sa["iterations"] == sb["iterations"] and sa["delta"] == sb["delta"]
    tr.close()


# ------------------------------------------------------------------------------------------------------------------------------
# 3. grey solve
# ------------------------------------------------------------------------------------------------------------------------------
SOLVE_N = [2, 15, 16, 17, 31, 33, 255, 256, 257, 511, 513, 2047, 2049, 4099]


def _check_solve(FL, coeff, h, j, g, st):
    """g == F'j of the returned j (matvec independent of convergence), and the reported residual is the true one.  FL: F as
    a longdouble array, or sparse."""
    jl = np.asarray(j, dtype=LD)
    g_ref = ref_matvec_t(FL, jl)
    mag = ref_matvec_t(_abs(FL), np.abs(jl))
    assert np.all(np.abs(np.asarray(g, dtype=LD) - g_ref) <= 2e-14 * mag + 1e-300)
    res = np.sqrt(np.sum((np.asarray(h, dtype=LD) - (jl - np.asarray(coeff, dtype=LD) * g_ref)) ** 2))
    scale = np.sqrt(np.sum((np.abs(h) + np.abs(jl) + np.abs(coeff) * mag) ** 2))
    assert res <= LD(st["residual"]) * (1 + LD(1e-6)) + LD(2e-14) * scale, (float(res), st["residual"])


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["row", "col", "csc"])
@pytest.mark.parametrize("n", SOLVE_N)
def test_solve_boundary_shapes(tracer, n, layout):
    F, coeff, h = grey_system(n, 500 + n, "csc" if layout == "csc" else "dense")
    arg = dict(F=F) if layout != "col" else dict(F=np.asfortranarray(F).T, col_major=True)
    Fd = F.toarray() if sp.issparse(F) else F
    FL = F if sp.issparse(F) else F.astype(LD)
    j_ref = np.linalg.solve(np.eye(n) - coeff[:, None] * Fd.T, h) if n <= 2049 else None
    for memory in sorted({1, 2, n, n + 5}):
        # GMRES(1) / GMRES(2) may stall before 1e-12 (and then say so); with memory >= n the Krylov space is complete
        j, g, st = tracer.solve_grey(coeff, h, memory=memory, max_iters=1000 if memory < n else 0, **arg)
        _check_solve(FL, coeff, h, j, g, st)
        assert st["converged"] == 1 or memory < n, (memory, st)
        if st["converged"]:
            assert st["residual"] <= 1.4901161193847656e-08 + 1e-12 * st["rhs_norm"]
            if j_ref is not None:
                assert np.abs(j - j_ref).max() <= 1e-9 * np.abs(j_ref).max()
    for it in (1, 2):                                        # far from the solution: the product must still be exact
        j, g, st = tracer.solve_grey(coeff, h, memory=50, max_iters=it, **arg)
        assert st["iterations"] == it or st["converged"] == 1
        _check_solve(FL, coeff, h, j, g, st)


@pytest.mark.gpu
def test_solve_from_resident_smoothed_matrix(tracer):
    n = 2049
    w, kw, _ = _dense_case(n, "F")
    Fs, _ = tracer.smooth(w, **kw)
    Fs = Fs.copy()
    _, coeff, h = grey_system(n, 77, "dense")
    j, g, st = tracer.solve_grey(coeff, h)
    assert st["converged"] == 1
    FL = Fs.astype(LD)
    _check_solve(FL, coeff, h, j, g, st)
    j_ref = np.linalg.solve(np.eye(n) - coeff[:, None] * Fs.T, h)
    assert np.abs(j - j_ref).max() <= 1e-9 * np.abs(j_ref).max()
    j2, g2, _ = tracer.solve_grey(coeff, h, F=Fs)              # the same padded layout uploaded: same kernels, same bits
    assert np.array_equal(j, j2) and np.array_equal(g, g2)
    j3, g3, st3 = tracer.solve_grey(coeff, h, max_iters=2)
    _check_solve(FL, coeff, h, j3, g3, st3)


# ------------------------------------------------------------------------------------------------------------------------------
# 4. count read-out at boundary N
# ------------------------------------------------------------------------------------------------------------------------------
def _band_mesh(rthx_mod, N):
    a, b = NDIV[N]
    rtm = rthx_mod.meshes.square_domain(kappa=1.0, n_bins=3, kappa_bins=[0.3, 1.0, 3.0], Ndiv=(a, b))
    assert rtm.num_elements == N
    return rtm


@pytest.mark.gpu
@pytest.mark.parametrize("N", sorted(NDIV))
def test_count_read_out_at_boundary_N(rthx_mod, cuda_lib, N):
    rtm = _band_mesh(rthx_mod, N)
    flat = rthx_mod.flatten_domain(rtm)
    tr = rthx_mod.DeviceTracer(flat, device=0)
    ns = flat.n_surfaces
    counts = tr.trace(max(40, 60_000 // N), seed=90 + N, bins=[0, 1, 2])["counts"].copy()
    for b in (2, 0, 1):
        c = counts[b]
        rs = c.sum(axis=1)                                   # exact: every row total is far below 2^64
        nz = c != 0
        nnz = int(nz.sum())
        rows, cols_ = np.nonzero(nz)                         # row-major order = CSR order
        row_ptr, cols, vals, fv = tr.counts_csr(b)
        assert np.array_equal(row_ptr, np.concatenate(([0], np.cumsum(nz.sum(axis=1)))))
        assert np.array_equal(cols, cols_) and np.array_equal(vals, c[nz])
        assert np.array_equal(fv, c[nz].astype(np.float64) * (1.0 / rs[rows].astype(np.float64)))
        colptr, rowval, cvals, cfv = tr.counts_csc(b, values=True)
        ct, ct_nz = c.T, nz.T
        cc, rr = np.nonzero(ct_nz)                           # column-major order = CSC order
        assert len(rowval) == nnz
        assert np.array_equal(colptr, np.concatenate(([0], np.cumsum(nz.sum(axis=0)))))
        assert np.array_equal(rowval, rr) and np.array_equal(cvals, ct[ct_nz])
        assert np.array_equal(cfv, ct[ct_nz].astype(np.float64) / rs[rr].astype(np.float64))
        nnz_d, chi = tr.counts_stats(b)
        F = np.zeros(c.shape)
        F[nz] = c[nz].astype(np.float64) / rs[rows].astype(np.float64)
        chi_ref = (F[:ns, ns:].sum() + F[ns:, :ns].sum()) / N
        assert nnz_d == nnz and abs(chi - chi_ref) <= 1e-12 * chi_ref
    if N == 1025:
        for rank in range(3):
            tr.trace(max(40, 60_000 // N), seed=90 + N, bins=[0, 1, 2], dense=False, emitter_rank=rank, emitter_world=3)
            for b in (0, 2):
                c = counts[b][rank::3]
                nz = c != 0
                rows = np.nonzero(nz)[0]
                rs = c.sum(axis=1)
                row_ptr, cols, vals, fv = tr.counts_csr(b)
                assert np.array_equal(row_ptr, np.concatenate(([0], np.cumsum(nz.sum(axis=1)))))
                assert np.array_equal(cols, np.nonzero(nz)[1]) and np.array_equal(vals, c[nz])
                assert np.array_equal(fv, c[nz].astype(np.float64) * (1.0 / rs[rows].astype(np.float64)))
    tr.close()


# ------------------------------------------------------------------------------------------------------------------------------
# 5. handle state
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_interleaved_calls_match_fresh_handles(rthx_mod, cuda_lib):
    """One handle runs CSC, sparse AP, CSR, dense AP, solve and CSC again (pooled buffers sized by different calls); every result
    is bit-identical to the same call on a fresh handle after the same trace."""
    rtm = rthx_mod.meshes.square_domain(11, kappa=1.5, n_bins=3, kappa_bins=[0.5, 1.5, 6.0])
    flat = rthx_mod.flatten_domain(rtm)
    N, ns = flat.n_elements, flat.n_surfaces
    w = weights(N, 5)
    coeff, rhs = np.random.default_rng(5).uniform(0, 0.6, N), np.random.default_rng(6).random(N) * 1e3

    def trace(tr):
        tr.trace(500, seed=95, bins=[0, 1, 2], dense=False)

    def csc2(tr):
        return tr.counts_csc(2)

    def sparse1(tr):
        Fs, st = tr.smooth_sparse(w[:ns + 1], n=ns + 1, bin=1)
        return Fs.indptr.copy(), Fs.indices.copy(), Fs.data.copy(), st["iterations"], st["delta"]

    def csr0(tr):
        return tr.counts_csr(0)

    def dense0(tr):
        Fs, st = tr.smooth(w, bin=0)
        return Fs.copy(), st["iterations"], st["delta"]

    def solve(tr):
        return tr.solve_grey(coeff, rhs)[:2]

    def csc2_julia(tr):
        return tr.counts_csc(2, values=True, index64=True, index_base=1)

    steps = [csc2, sparse1, csr0, dense0, solve, csc2_julia]
    shared = rthx_mod.DeviceTracer(flat, device=0)
    trace(shared)
    got = [step(shared) for step in steps]
    for k, step in enumerate(steps):
        fresh = rthx_mod.DeviceTracer(flat, device=0)
        trace(fresh)
        if step is solve:
            dense0(fresh)
        want = step(fresh)
        fresh.close()
        for a, b in zip(got[k], want):
            if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
                assert (a is None and b is None) or np.array_equal(a, b), step.__name__
            else:
                assert a == b, step.__name__
    cp, rv, cv, cf = got[5]
    cp0, rv0, _, cf0 = got[0]
    assert rv.dtype == np.int64 and np.array_equal(cp, cp0 + 1) and np.array_equal(rv, rv0 + 1) and np.array_equal(cf, cf0)
    assert cv.min() > 0
    shared.close()
