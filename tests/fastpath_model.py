"""numpy restatement of k_panel's fast path (distributedhouseholderqr.jl_b200/csrc/dhqr_kernels.cuh), stage by stage:
CholeskyQR2 (two Gram / Cholesky / triangular-solve passes with the kernel's guards) followed by Householder
reconstruction (LU of the top block of E - Q S with the signs picked on the fly, row-local solve below it), producing the
reference's storage (S:127-135: v scaled to |v|^2 = 2 in the lower trapezoid including the diagonal, R above, diag(R) in alpha).

Test infrastructure only (tests/test_fastpath_model.py): it pins on the CPU that the algorithm the kernel runs yields the
reflectors of the reference's column recurrences, and that the guards send ill-conditioned panels to the column path.
The triangular solves are the blocked form the kernel uses on the fp64 tensor pipe: 8-column blocks, explicitly inverted 8x8
diagonal blocks, products R_ab inv(R_bb) formed once.
"""
import numpy as np

IB = 32
SPREAD_MIN = 4e-3     # FAST_SPREAD_MIN of the kernel (its triangular solves run on the tensor pipe)


def blocked_trsm(X, R, dgi):
    """X <- X R^{-1} for upper-triangular R (IB x IB), dgi = 1 / diag(R); panel_trsm / trsm_dmma of the kernel."""
    X = np.array(X, dtype=np.float64, copy=True)
    nb = IB // 8
    Dv = []
    for b in range(nb):                                   # inverses of the diagonal blocks, one column per thread
        Rb = R[8 * b:8 * b + 8, 8 * b:8 * b + 8]
        inv = np.zeros((8, 8))
        for c in range(8):
            for i in range(7, -1, -1):
                s = 1.0 if i == c else 0.0
                for j in range(i + 1, 8):
                    s -= Rb[i, j] * inv[j, c]
                inv[i, c] = s * dgi[8 * b + i] if i <= c else 0.0
        Dv.append(inv)
    Wn = {(a, b): -(R[8 * a:8 * a + 8, 8 * b:8 * b + 8] @ Dv[b]) for b in range(nb) for a in range(b)}
    out = np.zeros_like(X)
    for b in range(nb):
        acc = X[:, 8 * b:8 * b + 8] @ Dv[b]
        for a in range(b):
            acc = acc + out[:, 8 * a:8 * a + 8] @ Wn[(a, b)]
        out[:, 8 * b:8 * b + 8] = acc
    return out


def cholesky_upper(G):
    """Right-looking upper Cholesky as in the kernel: returns (R, rinv, ok)."""
    g = np.array(G, dtype=np.float64, copy=True)
    R = np.zeros((IB, IB))
    rinv = np.zeros(IB)
    ok = True
    for j in range(IB):
        d = g[j, j]
        if not (d > 0.0) or not (d < 1e300):
            ok = False
            d = abs(d) + 1.0                                   # keep going with finite numbers; the result is discarded
        ri = 1.0 / np.sqrt(d)
        rinv[j] = ri
        R[j, j:] = g[j, j:] * ri
        R[j, j] = d * ri
        for i in range(j + 1, IB):
            g[i, i:] -= R[j, i] * R[j, i:]
    return R, rinv, ok


def fast_panel(P):
    """Returns (H, alpha, took_fast_path).  H, alpha are None when the guards ask for the column-by-column path."""
    P = np.array(P, dtype=np.float64)
    m, n = P.shape
    assert n == IB and m >= 2 * IB
    # pass 1
    R1, rinv1, ok = cholesky_upper(P.T @ P)
    d1 = np.diag(R1)
    if not ok or not (d1.min() > SPREAD_MIN * d1.max()):
        return None, None, False
    Q1 = blocked_trsm(P, R1, rinv1)
    # pass 2 with the orthogonality guard of the kernel
    G2 = Q1.T @ Q1
    if not np.all(np.abs(G2 - np.eye(IB)) <= 0.25 / IB):
        return None, None, False
    R2, rinv2, ok = cholesky_upper(G2)
    if not ok:
        return None, None, False
    Q = blocked_trsm(Q1, R2, rinv2)
    Rt = np.triu(R2 @ R1)
    # Householder reconstruction: LU of the top block of E - Q S, signs on the fly (CTA 0 of the kernel)
    Wt = Q[:IB, :].copy()
    Sg = np.zeros(IB)
    Ud = np.zeros(IB)
    for j in range(IB):
        w = Wt[j, j]
        Sg[j] = -1.0 if w > 0.0 else 1.0
        Ud[j] = 1.0 + abs(w)
        f = Sg[j] / Ud[j]
        Wt[j + 1:, j + 1:] += np.outer(f * Wt[j + 1:, j], Wt[j, j + 1:])
    rsq = 1.0 / np.sqrt(Ud)
    cl = -Sg / Ud
    # rows below the top block: V = M Rr^{-1}, Rr = diag(sqrt(Ud)) (I + diag(cl) striu(U))
    U = np.triu(Wt, 1)
    sq = Ud * rsq
    Rr = np.diag(sq) + (cl * sq)[:, None] * U
    H = np.zeros((m, IB))
    H[IB:, :] = blocked_trsm(Q[IB:, :], Rr, rsq)
    # top block: V below the diagonal, R above, alpha
    for i in range(IB):
        for j in range(IB):
            if i > j:
                H[i, j] = Wt[i, j] * rsq[j]
            elif i == j:
                H[i, j] = -Sg[j] * (Ud[j] * rsq[j])
            else:
                H[i, j] = Sg[i] * Rt[i, j]
    alpha = Sg * np.diag(Rt)
    return H, alpha, True


# ------------------------------------------------------------------------------------------------------------------------
# Design study for the next round (not what the kernel runs today): the two 32-step recurrences of the fast path in blocked
# form, 8-column blocks, so that only 8x8 diagonal blocks stay serial and everything else is a small GEMM (tensor pipe).
# ------------------------------------------------------------------------------------------------------------------------
def cholesky_upper_blocked(G, bs=8):
    """Upper Cholesky by bs-column blocks: serial factorisation of the diagonal block, row panel by a triangular solve with
    the explicitly inverted diagonal block, trailing update by a rank-bs product.  Returns (R, rinv, ok)."""
    g = np.array(G, dtype=np.float64, copy=True)
    n = g.shape[0]
    R = np.zeros((n, n))
    rinv = np.zeros(n)
    ok = True
    for k in range(0, n, bs):
        e = k + bs
        d = g[k:e, k:e].copy()
        Rd = np.zeros((bs, bs))
        for j in range(bs):                                     # serial part: bs steps on a bs x bs block
            p = d[j, j]
            if not (p > 0.0) or not (p < 1e300):
                ok = False
                p = abs(p) + 1.0
            ri = 1.0 / np.sqrt(p)
            rinv[k + j] = ri
            Rd[j, j:] = d[j, j:] * ri
            Rd[j, j] = p * ri
            for i in range(j + 1, bs):
                d[i, i:] -= Rd[j, i] * Rd[j, i:]
        R[k:e, k:e] = Rd
        if e < n:
            Rdinv = np.linalg.inv(Rd)                           # 8x8 triangular inverse (one thread per column in a kernel)
            R[k:e, e:] = Rdinv.T @ g[k:e, e:]                   # R12 = Rd^{-T} G12
            g[e:, e:] -= R[k:e, e:].T @ R[k:e, e:]              # G22 -= R12' R12
    return R, rinv, ok


def lu_signed_blocked(W, bs=8):
    """The top-block LU of Householder reconstruction (signs S_j = -sign(pivot) picked on the fly, pivots U_jj = 1 + |w_jj|,
    multipliers scaled by S_j / U_jj) in blocked right-looking form.  Returns (Wt, Sg, Ud) with the same meaning as the
    unblocked loop in fast_panel: strict upper part = frozen rows U, strict lower part = W_ij^(j)."""
    Wt = np.array(W, dtype=np.float64, copy=True)
    n = Wt.shape[0]
    Sg = np.zeros(n)
    Ud = np.zeros(n)
    for k in range(0, n, bs):
        e = k + bs
        for j in range(k, e):                                   # serial part, restricted to the block column / block row
            w = Wt[j, j]
            Sg[j] = -1.0 if w > 0.0 else 1.0
            Ud[j] = 1.0 + abs(w)
            f = Sg[j] / Ud[j]
            Wt[j + 1:, j + 1:e] += np.outer(f * Wt[j + 1:, j], Wt[j, j + 1:e])      # columns inside the block: all rows below
            Wt[j + 1:e, e:] += np.outer(f * Wt[j + 1:e, j], Wt[j, e:])              # rows inside the block: columns right of it
        if e < n:                                               # trailing update with the block's multipliers: one GEMM
            L = Wt[e:, k:e] * (Sg[k:e] / Ud[k:e])[None, :]      # -l_ij = f_j W_ij^(j)
            Wt[e:, e:] += L @ Wt[k:e, e:]
    return Wt, Sg, Ud
