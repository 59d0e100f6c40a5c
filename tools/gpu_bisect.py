"""Debug aid: the factorisation is deterministic by construction (fixed-order reductions), so two runs
must agree bitwise.  Compares sync=1 vs sync=0 runs and nb variants per 128-column panel."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import dhqr_b200 as D
dev = torch.device("cuda:0")
h = D.default_handle(0)
def run(m, n, sync, nb=0):
    h.set_option("sync", sync)
    A = D.colmajor_empty(m, n, dev); D.fill_uniform_(A, 0)
    al = torch.zeros(n, dtype=torch.float64, device=dev)
    D.householder_(A, al, nb)
    torch.cuda.synchronize()
    return A, al
def resid(A, al, m, n):
    R = torch.zeros(m, n, dtype=torch.float64, device=dev)
    R[:n] = torch.triu(A[:n], 1) + torch.diag(al)
    for k in range(((n - 1) // 128) * 128, -1, -128):
        kb = min(128, n - k)
        V = torch.tril(A[k:, k:k + kb])
        Tinv = torch.eye(kb, dtype=torch.float64, device=dev) + torch.triu(V.T @ V, 1)
        R[k:] -= V @ torch.linalg.solve_triangular(Tinv, V.T @ R[k:], upper=True)
    A0 = D.colmajor_empty(m, n, dev); D.fill_uniform_(A0, 0)
    return float(torch.linalg.norm(R - A0) / torch.linalg.norm(A0))
def cmp(tag, X, Y, n):
    d = (X[0] - Y[0]).abs()
    per = [float(d[:, k:k + 128].max()) for k in range(0, n, 128)]
    first = next((i for i, v in enumerate(per) if v > 0), None)
    print(f"{tag}: max diff {float(d.max()):.3e}; first differing panel {first}; per-panel {['%.1e' % v for v in per[:8]]}...", flush=True)
    if first is not None:
        k = first * 128
        dd = d[:, k:k + 128]
        idx = torch.nonzero(dd > 0)
        print(f"   panel {first}: {idx.shape[0]} differing entries; rows {int(idx[:,0].min())}..{int(idx[:,0].max())}, cols {int(idx[:,1].min())}..{int(idx[:,1].max())}", flush=True)
        rows = idx[:, 0]
        print("   row histogram (per 1024 rows):", torch.bincount(rows // 1024).tolist()[:40], flush=True)
        print("   col histogram:", torch.bincount(idx[:, 1]).tolist(), flush=True)
for (m, n) in [(16384, 2048), (32768, 4096)]:
    S1 = run(m, n, 1); print(f"{m}x{n} sync=1 resid {resid(*S1, m, n):.3e}", flush=True)
    S0 = run(m, n, 0); print(f"{m}x{n} sync=0 resid {resid(*S0, m, n):.3e}", flush=True)
    S0b = run(m, n, 0)
    cmp("sync1 vs sync0", S1, S0, n)
    cmp("sync0 vs sync0", S0, S0b, n)
    S1b = run(m, n, 1)
    cmp("sync1 vs sync1", S1, S1b, n)
