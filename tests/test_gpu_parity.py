"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C-ABI
(dhqr_b200 -> ctypes -> libdhqr.so), against the CPU oracle, the committed golden fixtures, LAPACK, and —
at BASELINE's full sizes — size-independent properties.

Tolerances (fp64, stated once):  max|H - H_oracle| <= 1e-10 (entries are O(1..sqrt(m)));
rel|alpha| <= 1e-12;  ||Q'b - oracle||_2/||b||_2 <= 1e-12;  ||QR - A||_F/||A||_F <= 1e-13;
normal-equation residual < 8x LAPACK's (the reference's own assertion, test/runtests.jl:62,81)."""
import ctypes as C
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "qr_*.npz")))
TOL_H, TOL_A, TOL_QTB, TOL_RES = 1e-10, 1e-12, 1e-12, 1e-13


@pytest.fixture(scope="module")
def D():
    import dhqr_b200
    assert torch.cuda.is_available()
    return dhqr_b200


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def vp(t):
    return C.c_void_p(t.data_ptr())


def sp():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def gpu_residual(D, A, alpha, A0):
    m, n = A.shape
    dev = A.device
    R = torch.zeros(m, n, dtype=torch.float64, device=dev)
    R[:n] = torch.triu(A[:n], 1) + torch.diag(alpha)
    for k in range(((n - 1) // 128) * 128, -1, -128):
        kb = min(128, n - k)
        V = torch.tril(A[k:, k:k + kb])
        Tinv = torch.eye(kb, dtype=torch.float64, device=dev) + torch.triu(V.T @ V, 1)       # T^{-1} = I + striu(V'V)
        R[k:] -= V @ torch.linalg.solve_triangular(Tinv, V.T @ R[k:], upper=True)
    return float(torch.linalg.norm(R - A0) / torch.linalg.norm(A0))


# ---------------------------------------------------------------------------------------------
def test_native_library_is_what_runs(D):
    # the .so must be loaded in-tree and be the sm_100a build; no fallback exists
    assert os.path.exists(D._lib.LIB_PATH)
    h = D.default_handle(0)
    assert h.get_option("sms") > 0
    l0 = h.launch_count()
    A = D.colmajor_empty(256, 64, "cuda:0")
    D.fill_uniform_(A, 0)
    D.qr_(A)
    torch.cuda.synchronize()
    assert h.launch_count() > l0


def test_fill_uniform_bit_exact(D, dev, oracle):
    A = D.colmajor_empty(257, 33, dev)
    D.fill_uniform_(A, 7, 3, 5)
    assert np.array_equal(A.cpu().numpy(), oracle.np_uniform(7, 257, 33, 3, 5))


def test_partialdot_suffixes(D, dev):
    # test/partialdot.jl:11-22 (real analogue): N = 1..20, every suffix, vs dot
    g = torch.Generator().manual_seed(0)
    for N in range(1, 21):
        a = torch.rand(N, dtype=torch.float64, generator=g).to(dev)
        b = torch.rand(N, dtype=torch.float64, generator=g).to(dev)
        for i in range(N):
            ref = float(a[i:] @ b[i:])
            assert D.partialdot(a, b, range(i, N)) == pytest.approx(ref, rel=1e-13)


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p) for p in GOLD])
@pytest.mark.parametrize("nb", [0, 1])
def test_golden_fixtures(D, dev, path, nb):
    g = np.load(path)
    A = D.to_colmajor(g["A"], dev)
    H = D.qr_(A, nb=nb)
    assert np.abs(A.cpu().numpy() - g["H"]).max() < TOL_H
    assert np.abs(H.α.cpu().numpy() - g["alpha"]).max() < TOL_A * np.abs(g["alpha"]).max()
    b = torch.from_numpy(g["b"]).to(dev)
    qtb = D.apply_qt_(b.clone(), A).cpu().numpy()
    assert np.linalg.norm(qtb - g["qtb"]) < TOL_QTB * np.linalg.norm(g["b"])
    x = D.ldiv(H, b).cpu().numpy()
    assert np.abs(x - g["x"]).max() < 1e-9 * max(1.0, np.abs(g["x"]).max())
    assert torch.equal(b.cpu(), torch.from_numpy(g["b"]))           # \ does not modify b (S:318)


# the reference's own sizes (test/runtests.jl:42) and the BASELINE configs that fit a quick CPU oracle run
@pytest.mark.parametrize("mn", [(110, 100), (220, 200), (440, 400), (880, 800), (1100, 1000), (2200, 2000),
                                (4400, 4000), (1024, 128), (8192, 1024)])
def test_qr_and_solve_against_oracle(D, dev, oracle, coracle, mn):
    m, n = mn
    A0 = coracle.fill_uniform(0, m, n)
    b = oracle.np_uniform(1, m, 1)[:, 0].copy()
    Href = A0.copy(order="F")
    Href, aref = coracle.qr(Href)
    A = D.colmajor_empty(m, n, dev)
    D.fill_uniform_(A, 0)
    H = D.qr_(A)
    Hg, ag = A.cpu().numpy(), H.α.cpu().numpy()
    assert np.abs(Hg - Href).max() < TOL_H
    assert np.abs(ag - aref).max() < TOL_A * np.abs(aref).max()
    assert oracle.qr_residual(A0, np.asfortranarray(Hg), ag) < TOL_RES
    bt = torch.from_numpy(b).to(dev)
    qtb = D.apply_qt_(bt.clone(), A).cpu().numpy()
    assert np.linalg.norm(qtb - coracle.apply_qt(Href, b)) < TOL_QTB * np.linalg.norm(b)
    x = D.ldiv(H, bt).cpu().numpy()
    xr = coracle.ldiv(Href, aref, b)
    stdliberr = oracle.normal_eq_residual(A0, oracle.lapack_lstsq(A0, b), b)       # T:49-51
    # T:62: < 8x the stdlib's residual.  On U[0,1) data at 4400 x 4000 the reference's OWN recurrences (the oracle) sit at
    # 8-14x LAPACK's, depending on LAPACK's thread count; where the reference itself misses its bound, the bar is "no worse
    # than the reference algorithm on the same input"
    bound = max(8 * stdliberr, 1.5 * oracle.normal_eq_residual(A0, xr, b))
    assert oracle.normal_eq_residual(A0, x, b) < bound
    assert np.abs(x - xr).max() < 1e-9 * np.abs(xr).max()


@pytest.mark.parametrize("mn", [(1024, 128), (8192, 1024), (1001, 37)])
def test_unblocked_path_config2(D, dev, oracle, coracle, mn):
    # BASELINE config 2: nb = 1, one reflector per step like S:127-144, TMA-staged column tiles
    m, n = mn
    A0 = coracle.fill_uniform(2, m, n)
    Href = A0.copy(order="F")
    Href, aref = coracle.qr(Href)
    A = D.to_colmajor(A0, dev)
    H = D.qr_(A, nb=1)
    assert np.abs(A.cpu().numpy() - Href).max() < TOL_H
    assert np.abs(H.α.cpu().numpy() - aref).max() < TOL_A * np.abs(aref).max()


@pytest.mark.parametrize("case", [(1000, 37, 0), (1001, 37, 0), (999, 130, 1), (515, 259, 3), (64, 64, 0), (33, 33, 0),
                                  (300, 1, 0), (2, 1, 0), (1, 1, 0)])
@pytest.mark.parametrize("nb", [0, 32, 64, 96])
def test_ragged_shapes_and_leading_dimensions(D, dev, oracle, coracle, case, nb):
    # odd m (unaligned TMA sources -> generic path), n not a multiple of the panel width, lda > m, m == n
    m, n, extra = case
    A0 = coracle.fill_uniform(9, m, n)
    Href = A0.copy(order="F")
    Href, aref = coracle.qr(Href)
    A = D.colmajor_empty(m, n, dev, lda=m + extra)
    A.copy_(torch.from_numpy(A0))
    H = D.qr_(A, nb=nb)
    assert np.abs(A.cpu().numpy() - Href).max() < TOL_H
    assert np.abs(H.α.cpu().numpy() - aref).max() < TOL_A * max(np.abs(aref).max(), 1e-300)
    b = oracle.np_uniform(10, m, 1)[:, 0].copy()
    x = D.ldiv(H, torch.from_numpy(b).to(dev)).cpu().numpy()
    xr = coracle.ldiv(Href, aref, b)
    assert np.abs(x - xr).max() < 1e-8 * max(1.0, np.abs(xr).max())


def test_empty_and_degenerate_inputs(D, dev):
    A = D.colmajor_empty(5, 0, dev)
    H = D.qr_(A)
    assert H.α.numel() == 0                                            # n == 0: nothing to do
    # zero column: f = 1/sqrt(0) = Inf -> NaN, not an error (S:131); mirrored, not fixed
    Z = torch.zeros(64, 3, dtype=torch.float64)
    Z[:, 0] = 1.0
    Z[:, 2] = torch.arange(64, dtype=torch.float64)
    A = D.to_colmajor(Z, dev)
    D.qr_(A)
    assert torch.isnan(A).any()
    with pytest.raises(D._lib.DhqrError) as e:                        # n > m is rejected (-3), reference would go out of bounds
        D.qr_(D.colmajor_empty(3, 5, dev))
    assert e.value.code == -3


def test_exact_zero_pivot_is_a_documented_divergence(D, dev, oracle):
    # alphafactor(0) = -sign(0) = 0 (S:8): with an exactly zero pivot the reference sets alpha = 0, its "reflector" has |v|^2 = 1
    # and the factorisation is garbage (later a division by zero).  The unblocked path mirrors that literally; the blocked paths
    # (Householder reconstruction picks the sign of a zero pivot as +) return a VALID factorisation instead - pinned here.
    for m, n in ((300, 40), (1024, 256)):                     # narrow chain / wide chain
        A0 = oracle.np_uniform(17, m, n)
        A0[0, 0] = 0.0
        A = D.to_colmajor(A0, dev)
        H = D.qr_(A)
        Hg, ag = A.cpu().numpy(), H.α.cpu().numpy()
        assert np.isfinite(Hg).all() and oracle.qr_residual(A0, np.asfortranarray(Hg), ag) < TOL_RES
        assert abs(abs(ag[0]) - np.linalg.norm(A0[:, 0])) < 1e-12 * np.linalg.norm(A0[:, 0])
        Hr, ar = oracle.np_qr(A0)                                 # the reference's recurrences on the same input
        assert ar[0] == 0.0 and not oracle.qr_residual(A0, Hr, ar) < 1e-3
        A1 = D.to_colmajor(A0, dev)
        H1 = D.qr_(A1, nb=1)                                      # the literal column loop reproduces the reference
        assert float(H1.α[0]) == 0.0


def test_multiple_right_hand_sides(D, dev, oracle, coracle):
    m, n, k = 700, 90, 5
    A0 = coracle.fill_uniform(4, m, n)
    B0 = oracle.np_uniform(5, m, k)
    Href = A0.copy(order="F")
    Href, aref = coracle.qr(Href)
    A = D.to_colmajor(A0, dev)
    H = D.qr_(A)
    X = D.ldiv(H, torch.from_numpy(B0).to(dev)).cpu().numpy()
    for j in range(k):
        xr = coracle.ldiv(Href, aref, B0[:, j].copy())
        assert np.abs(X[:, j] - xr).max() < 1e-9 * np.abs(xr).max()


def test_apply_q_is_the_inverse_sweep(D, dev, oracle, coracle):
    # Q b = H_1 ... H_n b (SURVEY 8f-3: the factorisation as an operator): inverts apply_qt_, reproduces A = Q R column by
    # column, and matches the numpy sweep of the oracle's reflectors
    for m, n in [(300, 37), (1100, 1000), (4096, 640)]:
        A0 = coracle.fill_uniform(6, m, n)
        Href = A0.copy(order="F")
        Href, aref = coracle.qr(Href)
        A = D.to_colmajor(A0, dev)
        H = D.qr_(A)
        B0 = oracle.np_uniform(7, m, 3)
        B = D.to_colmajor(B0, dev)
        D.apply_qt_(B, A)
        D.apply_q_(B, A)
        assert np.abs(B.cpu().numpy() - B0).max() < 1e-12 * np.abs(B0).max() * np.sqrt(m)
        b = B0[:, 0].copy()
        w = b.copy()
        for j in range(n - 1, -1, -1):                                   # H_1 (H_2 (... H_n b))
            v = Href[j:, j]
            w[j:] -= v * (v @ w[j:])
        qb = D.apply_q_(torch.from_numpy(b).to(dev), A).cpu().numpy()
        assert np.linalg.norm(qb - w) < TOL_QTB * np.linalg.norm(b)
        R = torch.zeros(m, 4, dtype=torch.float64)
        cols = [0, 1, n // 2, n - 1]
        for q, c in enumerate(cols):
            R[:c, q] = torch.from_numpy(Href[:c, c])
            R[c, q] = aref[c]
        QR = D.apply_q_(D.to_colmajor(R, dev), A).cpu().numpy()
        assert np.abs(QR - A0[:, cols]).max() < 1e-12 * np.sqrt(m)


def test_bitwise_determinism(D, dev):
    # fixed-order reductions everywhere: two runs must agree bit for bit (this is what exposed the TMA WAR race)
    outs = []
    for _ in range(3):
        A = D.colmajor_empty(16384, 1024, dev)
        D.fill_uniform_(A, 3)
        H = D.qr_(A)
        outs.append((A.clone(), H.α.clone()))
    for A, al in outs[1:]:
        assert torch.equal(A, outs[0][0]) and torch.equal(al, outs[0][1])


def test_lookahead_and_serial_schedules_agree(D, dev, oracle):
    # the look-ahead schedule regroups the trailing updates (other split-K partitions) but applies the same
    # reflectors in the same order: both schedules must agree to rounding and meet the same tolerances
    h = D.default_handle(0)
    m, n = 6000, 900
    res = {}
    try:
        for la in (0, 1):
            h.set_option("lookahead", la)
            A = D.colmajor_empty(m, n, dev)
            D.fill_uniform_(A, 5)
            H = D.qr_(A)
            torch.cuda.synchronize()
            res[la] = (A.cpu().numpy(), H.α.cpu().numpy())
    finally:
        h.set_option("lookahead", 1)
    assert np.abs(res[0][0] - res[1][0]).max() < 1e-11
    assert np.abs(res[0][1] - res[1][1]).max() < TOL_A * np.abs(res[0][1]).max()
    A0 = oracle.np_uniform(5, m, n)
    for la in (0, 1):
        assert oracle.qr_residual(A0, np.asfortranarray(res[la][0]), res[la][1]) < TOL_RES


def test_block_reflector_kernels(D, dev, oracle):
    # gemm_vta + tinv + ymake + gemm_cvy in isolation against torch fp64 on genuine Householder blocks
    h = D.default_handle(0)
    for rows, nbp, ncols, row_lo, ex in [(256, 32, 64, 0, 0), (1000, 32, 96, 7, 0), (999, 32, 33, 0, 1), (512, 128, 128, 0, 0),
                                         (4100, 100, 300, 5, 0), (4099, 64, 77, 3, 1), (33000, 128, 1000, 0, 0)]:
        Hp, _ = oracle.np_qr(oracle.np_uniform(11, rows - row_lo, nbp))
        V = torch.zeros(rows, nbp, dtype=torch.float64)
        V[row_lo:] = torch.from_numpy(np.tril(Hp))
        Cm = torch.rand(rows, ncols, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
        dV = D.to_colmajor(V, dev)
        dC = D.colmajor_empty(rows, ncols, dev, lda=rows + ex)
        dC.copy_(Cm)
        nbk = 32 if nbp <= 32 else 128
        dL = torch.zeros(nbk * nbk, dtype=torch.float64, device=dev)
        D._lib.call("dhqr_k_block_reflector_f64", h.raw, rows, nbp, vp(dV), rows, row_lo, ncols, vp(dC), rows + ex, vp(dL), sp())
        Vd, Cd = V.to(dev), Cm.to(dev)
        L = torch.eye(nbp, dtype=torch.float64, device=dev) + torch.tril(Vd.T @ Vd, -1)
        Linv = torch.linalg.solve_triangular(L, torch.eye(nbp, dtype=torch.float64, device=dev), upper=False)
        Cexp = Cd - Vd @ (Linv @ (Vd.T @ Cd))
        Cexp[:row_lo] = Cd[:row_lo]
        assert float((dL.view(nbk, nbk).T[:nbp, :nbp] - Linv).abs().max()) < 1e-12
        assert float((dC - Cexp).abs().max() / Cexp.abs().max()) < 1e-13


def test_panel_kernel(D, dev, oracle):
    h = D.default_handle(0)
    for rows, ncols in [(64, 32), (40, 32), (32, 32), (300, 7), (5000, 32), (33000, 32), (65536, 32)]:
        A = oracle.np_uniform(1, rows, ncols)
        Href, aref = oracle.np_qr(A)
        dP = D.to_colmajor(A, dev)
        dal = torch.zeros(ncols, dtype=torch.float64, device=dev)
        D._lib.call("dhqr_k_panel_f64", h.raw, rows, ncols, vp(dP), rows, vp(dal), sp())
        assert np.abs(dP.cpu().numpy() - Href).max() < 1e-11
        assert np.abs(dal.cpu().numpy() - aref).max() < TOL_A * np.abs(aref).max()


def test_panel_fast_path_and_fallback(D, dev, oracle):
    # CholeskyQR2 + Householder reconstruction must give the reference's reflectors; ill-conditioned, zero and NaN
    # panels must take the column-by-column fallback (decided on the device) and still match the oracle
    h = D.default_handle(0)
    rows = 4096

    def run(P):
        dP = D.to_colmajor(P, dev)
        dal = torch.zeros(32, dtype=torch.float64, device=dev)
        D._lib.call("dhqr_k_panel_f64", h.raw, rows, 32, vp(dP), rows, vp(dal), sp())
        torch.cuda.synchronize()
        return dP.cpu().numpy(), dal.cpu().numpy()

    P = oracle.np_uniform(21, rows, 32)
    Href, aref = oracle.np_qr(P)
    f0, b0 = h.get_option("panels_fast"), h.get_option("panels_fallback")
    Hf, af = run(P)
    assert h.get_option("panels_fast") == f0 + 1 and h.get_option("panels_fallback") == b0
    try:
        h.set_option("panel_fast", 0)
        Hs, as_ = run(P)
    finally:
        h.set_option("panel_fast", 1)
    for Hx, ax in ((Hf, af), (Hs, as_)):
        assert np.abs(Hx - Href).max() < 1e-11 and np.abs(ax - aref).max() < TOL_A * np.abs(aref).max()
    # nearly dependent columns: kappa ~ 1e9 > the guard -> fallback, result as accurate as the reference recurrences
    Pi = P.copy()
    Pi[:, 7] = Pi[:, 3] + 1e-9 * oracle.np_uniform(22, rows, 1)[:, 0]
    Hr2, ar2 = oracle.np_qr(Pi)
    b1 = h.get_option("panels_fallback")
    Hi, ai = run(Pi)
    assert h.get_option("panels_fallback") == b1 + 1
    assert oracle.qr_residual(Pi, np.asfortranarray(Hi), ai) < TOL_RES
    assert np.abs(ai - ar2).max() < 1e-6 * np.abs(ar2).max()          # alpha_7 is O(1e-9): relative accuracy limited by kappa
    # moderately ill-conditioned (kappa ~ 1e6): whichever path the guards pick, the factorisation must be backward stable
    Pm = P.copy()
    Pm[:, 9] = Pm[:, 2] + 1e-6 * oracle.np_uniform(23, rows, 1)[:, 0]
    Hm, am = run(Pm)
    Hr3, ar3 = oracle.np_qr(Pm)
    assert oracle.qr_residual(Pm, np.asfortranarray(Hm), am) < TOL_RES
    assert np.abs(am - ar3).max() < 1e-8 * np.abs(ar3).max()
    # zero column: the reference gives f = Inf -> NaN (S:131); the fast path must not "fix" that
    Pz = P.copy()
    Pz[:, 5] = 0.0
    Hz, _ = run(Pz)
    assert np.isnan(Hz).any()


def test_host_buffer_entry_points(D, oracle, coracle):
    # (4096, 2176) takes the two-half pipeline of dhqr_qr_host_f64 (right half uploads while the left half is factored)
    for m, n in [(1024, 128), (1001, 37), (4096, 2176)]:
        A0 = coracle.fill_uniform(3, m, n)
        Href = A0.copy(order="F")
        Href, aref = coracle.qr(Href)
        A = A0.copy(order="F")
        H = D.qr_(A)                                                   # numpy in -> dhqr_qr_host_f64
        assert H.A is A and np.abs(A - Href).max() < TOL_H
        b = oracle.np_uniform(4, m, 1)[:, 0].copy()
        b_keep = b.copy()
        x = D.ldiv(H, b)
        xr = coracle.ldiv(Href, aref, b)
        assert np.abs(x - xr).max() < 1e-9 * np.abs(xr).max() and np.array_equal(b, b_keep)


def test_aliasing_and_repeatable_solve(D, dev, oracle):
    # qr! aliases its input (H.A === A, S:314); \ may be called repeatedly on one factorisation (S:317-321)
    A = D.colmajor_empty(500, 60, dev)
    D.fill_uniform_(A, 0)
    H = D.qr_(A)
    assert H.A is A
    b = torch.rand(500, dtype=torch.float64, device=dev)
    x1, x2 = D.ldiv(H, b), D.ldiv(H, b)
    assert torch.equal(x1, x2)


# ---- BASELINE's full sizes through size-independent properties -------------------------------------
@pytest.mark.parametrize("mn", [(32768, 4096)])
def test_full_size_properties(D, dev, coracle, mn):
    m, n = mn
    A0 = D.colmajor_empty(m, n, dev)
    D.fill_uniform_(A0, 0)
    A = A0.clone()
    H = D.qr_(A)
    assert gpu_residual(D, A, H.α, A0) < TOL_RES                       # ||QR - A|| / ||A||
    # |v_j|^2 == 2 for every reflector (S:131-135)
    nrm = (torch.tril(A) ** 2).sum(0)
    assert float((nrm - 2.0).abs().max()) < 1e-12
    # Q' is orthogonal: ||Q'b|| == ||b||;  x solves the normal equations
    b = torch.rand(m, dtype=torch.float64, device=dev)
    qtb = D.apply_qt_(b.clone(), A)
    assert abs(float(torch.linalg.norm(qtb) / torch.linalg.norm(b)) - 1.0) < 1e-13
    x = D.ldiv(H, b)
    r = A0.T @ (A0 @ x) - A0.T @ b
    x_ref = torch.linalg.lstsq(A0, b.unsqueeze(1)).solution[:, 0]
    r_ref = A0.T @ (A0 @ x_ref) - A0.T @ b
    assert float(torch.linalg.norm(r)) < 8 * float(torch.linalg.norm(r_ref))   # T:62 with cuSOLVER as "stdlib"
    # H[:, :k] and alpha[:k] depend on A[:, :k] only: the C oracle on the leading 256 columns pins the full-size run
    k = 256
    Hk = coracle.fill_uniform(0, m, k)
    Hk, ak = coracle.qr(Hk)
    assert np.abs(A[:, :k].cpu().numpy() - Hk).max() < TOL_H
    assert np.abs(H.α[:k].cpu().numpy() - ak).max() < TOL_A * np.abs(ak).max()
    # LAPACK (cuSOLVER geqrf) at full size through the storage-format identity alpha = diag(R), triu(H,1) = triu(R,1)
    Rl = torch.geqrf(A0)[0]
    scale = float(Rl[:n].abs().max())
    assert float((torch.diagonal(Rl[:n]) - H.α).abs().max()) < 1e-11 * scale
    assert float((torch.triu(Rl[:n], 1) - torch.triu(A[:n], 1)).abs().max()) < 1e-10 * scale
    del Rl
    # unblocked and blocked paths agree (linearity of the algorithm in storage): compare alpha on a slice
    A2 = A0[:, :256].clone()
    A3 = D.colmajor_empty(m, 256, dev)
    A3.copy_(A2)
    H3 = D.qr_(A3, nb=1)
    assert float((H3.α - H.α[:256]).abs().max() / H.α.abs().max()) < TOL_A


# ---- bench.py --dump-outputs: what the timed qr! handed back -----------------------------------------
def test_bench_dump_outputs_are_the_factorisation(tmp_path, coracle):
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    m, n = 2048, 256
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "3", "--m", str(m),
                          "--n", str(n), "--no-e2e", "--no-cpu", "--no-solve", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    A, alpha = np.load(tmp_path / "A.npy"), np.load(tmp_path / "alpha.npy")
    assert A.shape == (m, n) and A.dtype == np.float64 and alpha.shape == (n,)    # small enough to be written whole
    Href, aref = coracle.qr(coracle.fill_uniform(0, m, n))
    assert np.abs(A - Href).max() < TOL_H
    assert np.abs(alpha - aref).max() < TOL_A * np.abs(aref).max()
