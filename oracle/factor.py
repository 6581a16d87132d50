"""Multilevel HIF factors computed on the host from this repository alone (numpy / scipy): the factor
producer of bench.py and of the tests that need factors larger than the committed goldens.

Every level has the structure of a hif::Prec and the layout of the level dicts the device backend is
attached with (hifir_b200.make_level_structs):

  * symmetric scaling s = t = |a_ii|^-1/2 (rows without a usable diagonal: the row's largest entry);
  * a split into B (kept) and the deferred set: every row whose scaled diagonal vanishes (the pressure
    rows of a saddle-point system) plus an independent set of the others, chosen with seeded random
    priorities (one Luby round).  p = q = [B in original order, deferred];
  * B = (I + L_B) D_B (I + U_B) by D-ILU: L_B and U_B keep B's strictly lower / upper parts and the
    pivots d_i = b_ii - sum_{j<i} b_ij b_ji / d_j give the product B's diagonal;
  * E, F = the off-diagonal blocks, and the next level is the sparse approximate Schur complement
    S = C - E D_B^-1 F + E D_B^-1 R_B D_B^-1 F, R_B = B - diag(B) (B^-1 to first order);
  * once S has at most DENSE_MAX rows it becomes the dense last level, factorized by QR with column
    pivoting (LAPACK dgeqp3); its numerical rank drops the directions of a singular S (pure Neumann).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl
import scipy.sparse as sp

NAME = "multilevel D-ILU, independent-set Schur levels, dense QRCP last level"
NAME_KEY = "dilu_is_qrcp_v1"  # names these factors in on-disk caches; change it with the algorithm
DENSE_MAX = 1500
MAX_LEVELS = 12
SEED = 20260101
RANK_TOL = 1e-12  # |R_kk| <= RANK_TOL |R_00|: beyond the numerical rank of the dense level


def _segments(starts, counts):
    """positions starts[r] .. starts[r] + counts[r] - 1 of every r, concatenated"""
    total = int(counts.sum())
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    return np.repeat(starts - first, counts) + np.arange(total)


def dilu_pivots(B):
    """D-ILU pivots of B (CSR): d_i = b_ii - sum_{j<i} b_ij b_ji / d_j.  Rows are processed front by
    front of their dependency graph, each front in one vectorised step."""
    n = B.shape[0]
    P = sp.tril(B, -1, format="csr").multiply(sp.triu(B, 1, format="csr").T).tocsr()
    P.eliminate_zeros()
    P.sort_indices()
    succ = P.T.tocsr()
    pending = np.diff(P.indptr).astype(np.int64)
    d = B.diagonal().astype(np.float64)
    front = np.flatnonzero(pending == 0)
    done = 0
    while front.size:
        done += front.size
        cnt = P.indptr[front + 1] - P.indptr[front]
        pos = _segments(P.indptr[front], cnt)
        if pos.size:
            d[front] -= np.bincount(np.repeat(np.arange(front.size), cnt),
                                    weights=P.data[pos] / d[P.indices[pos]], minlength=front.size)
        spos = _segments(succ.indptr[front], succ.indptr[front + 1] - succ.indptr[front])
        nxt, k = np.unique(succ.indices[spos], return_counts=True)
        pending[nxt] -= k
        front = nxt[pending[nxt] == 0]
    assert done == n
    return d


def _deferred(A, rng):
    """rows with a vanishing (scaled) diagonal, plus one Luby round of an independent set of the others"""
    n = A.shape[0]
    weak = np.abs(A.diagonal()) <= 1e-8
    prio = np.where(weak, -1.0, rng.random(n))
    rows = np.repeat(np.arange(n), np.diff(A.indptr))
    nb = np.where(A.indices == rows, -1.0, prio[A.indices])
    nbmax = np.full(n, -1.0)
    np.maximum.at(nbmax, rows, nb)
    linked = np.bincount(rows, weights=(A.indices != rows) & (A.data != 0), minlength=n) > 0
    return weak | (linked & (prio > nbmax))  # a node without neighbours gains nothing from deferral


def _ccs(T, dtype):
    T = sp.csc_matrix(T)
    T.sort_indices()
    return T.shape[0], T.shape[1], T.indptr.astype(np.int64), T.indices.astype(np.int32), T.data.astype(dtype)


def _level(A, rng, dtype):
    """one level of A (CSR): returns (level dict, Schur complement CSR)"""
    n = A.shape[0]
    absA = abs(A)
    rowmax = np.zeros(n)
    np.maximum.at(rowmax, np.repeat(np.arange(n), np.diff(A.indptr)), absA.data)
    diag = np.abs(A.diagonal())
    s = 1.0 / np.sqrt(np.where(diag > 1e-12 * rowmax, diag, rowmax))
    Ah = sp.csr_matrix(sp.diags(s) @ A @ sp.diags(s))
    gamma = _deferred(Ah, rng)
    while True:
        perm = np.concatenate([np.flatnonzero(~gamma), np.flatnonzero(gamma)])
        m = int((~gamma).sum())
        Ap = Ah[perm][:, perm].tocsr()
        Bm = Ap[:m, :m].tocsr()
        d = dilu_pivots(Bm)
        small = np.abs(d) <= 1e-6 * np.abs(Bm.diagonal())
        if not small.any():
            break
        gamma[perm[:m][small]] = True  # tiny pivots: deferred to the next level, as HIF does
    E, F, C = Ap[m:, :m], Ap[:m, m:], Ap[m:, m:]
    Dinv = sp.diags(1.0 / d)
    ED, DF = E @ Dinv, Dinv @ F
    S = sp.csr_matrix(C - ED @ F + ED @ (Bm - sp.diags(Bm.diagonal())) @ DF)
    S.sort_indices()
    perm = perm.astype(np.int32)
    inv = np.argsort(perm).astype(np.int32)
    lev = dict(m=m, n=n, dense_n=0, dense_rank=0, has_symm_dense=0,
               L=_ccs(sp.tril(Bm, -1) @ Dinv, dtype), U=_ccs(Dinv @ sp.triu(Bm, 1), dtype),
               E=_ccs(E, dtype), F=_ccs(F, dtype), d=d.astype(dtype), s=s.astype(dtype), t=s.astype(dtype),
               p=perm, p_inv=inv, q=perm, q_inv=inv)
    return lev, S


def multilevel_levels(A, dtype=np.float64):
    """Multilevel factors of A = (n, indptr, indices, vals) as a list of level dicts; dtype=float32
    stores single-precision factors (computed in double) for the lhfs* / lhfsd* entry points."""
    n, indptr, indices, vals = A
    M = sp.csr_matrix((vals, indices, indptr), shape=(n, n))
    M.sort_indices()
    rng = np.random.default_rng(SEED)
    levels = []
    for _ in range(MAX_LEVELS):
        lev, S = _level(M, rng, dtype)
        levels.append(lev)
        nm = S.shape[0]
        if nm == 0:  # nothing deferred: this level is the last (m == n)
            return levels
        if nm <= DENSE_MAX:
            (qr, tau), r, piv = sl.qr(S.toarray(), mode="raw", pivoting=True)
            rd = np.abs(np.diag(r))
            rank = int((rd > RANK_TOL * rd[0]).sum())
            lev.update(dense_n=nm, dense_rank=rank, qr_mat=np.asfortranarray(qr).ravel(order="F").astype(dtype),
                       qr_tau=tau.astype(dtype), qr_jpvt=(piv + 1).astype(np.int32))
            return levels
        M = S
    raise RuntimeError(f"Schur complement still has {M.shape[0]} rows after {MAX_LEVELS} levels")
