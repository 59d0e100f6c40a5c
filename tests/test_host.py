"""Host-side mirror of the reference interface: layout and partition logic (no GPU needed)."""
import numpy as np
import pytest
import torch

import dhqr_b200 as D


def test_splits_match_darray_default_distribution():
    # DistributedArrays defaultdist: even chunks, remainder to the first blocks (T:71 uses (1, nworkers()))
    assert D.splits(2, 100) == [0, 50, 100]
    assert D.splits(4, 4096) == [0, 1024, 2048, 3072, 4096]
    assert D.splits(3, 10) == [0, 4, 7, 10]
    assert D.splits(8, 8192)[-1] == 8192 and len(D.splits(8, 8192)) == 9
    for P in range(1, 9):
        b = D.splits(P, 103)
        assert b[0] == 0 and b[-1] == 103 and all(0 <= b[i + 1] - b[i] <= 103 // P + 1 for i in range(P))


def test_colmajor_helpers_cpu():
    A = D.colmajor_empty(5, 3, device="cpu")
    assert A.shape == (5, 3) and A.stride() == (1, 5)
    B = D.colmajor_empty(5, 3, device="cpu", lda=8)
    assert B.stride() == (1, 8)
    x = np.arange(12.0).reshape(4, 3)
    C = D.to_colmajor(x, device="cpu")
    assert C.stride() == (1, 4) and np.array_equal(C.numpy(), x)


def test_local_column_block_indexing():
    # LocalColumnBlock (S:26-40): global column j lives at local column j - dj
    Al = D.to_colmajor(np.arange(20.0).reshape(4, 5), device="cpu")
    blk = D.LocalColumnBlock(Al, 10, range(10, 15))
    assert torch.equal(blk.global_col(12), Al[:, 2])


def test_alphafactor():
    assert D.alphafactor(3.0) == -1.0 and D.alphafactor(-2.0) == 1.0 and D.alphafactor(0.0) == 0.0


def test_rejects_row_major_and_wrong_dtype():
    from dhqr_b200.api import _lda
    with pytest.raises(ValueError):
        _lda(torch.zeros(4, 3, dtype=torch.float64))            # row-major
    with pytest.raises(TypeError):
        _lda(D.colmajor_empty(4, 3, device="cpu").float())


def test_bench_reference_arm_is_stable_under_torchrun_env():
    """The CPU arm sizes its OpenMP team from the affinity mask (torch.distributed.run exports OMP_NUM_THREADS=1, which voided
    the round-1 ratios at N > 1), samples the whole column sweep at a fixed stride, and names the same config as the GPU arm."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    phys, logical = bench.host_cores()
    assert 1 <= phys <= logical == len(os.sched_getaffinity(0))
    assert bench.cpu_stride(32768, 4096) == 8 and bench.cpu_stride(1024, 128) == 1
    assert bench.make_config(32768, 4096, 4) == bench.make_config(32768, 4096, 4)
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--m", "2048", "--n", "256",
                          "--steps", "2", "--warmup", "1"], env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["cores"] == phys and line["value"] > 0
    assert line["config"] == bench.make_config(2048, 256, 2)
    assert line["e2e"]["value"] == line["value"] and line["cpu_baseline"]["kind"] == "port"
    # ranks other than 0 exit without work
    out1 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--m", "2048", "--n", "256",
                           "--steps", "1", "--warmup", "0"], env=dict(env, RANK="1"), capture_output=True, text=True, timeout=60)
    assert out1.returncode == 0 and out1.stdout.strip() == ""


def test_strided_sample_is_the_genuine_column_step():
    """dhqr_oracle_qr_steps_strided at stride 1 is the full factorisation; at stride s it performs exactly the flops of the
    sampled steps (what bench.py divides by the measured time)."""
    import os, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "oracle"))
    import dhqr_oracle as O
    co = O.COracle()
    A = co.fill_uniform(1, 600, 90)
    H, al = co.qr(A.copy(order="F"), 2)
    B = A.copy(order="F")
    al2, fl = co.qr_steps_strided(B, 0, 1, 2)
    assert np.array_equal(B, H) and np.array_equal(al, al2)
    m, n = A.shape
    _, fl3 = co.qr_steps_strided(A.copy(order="F"), 2, 7, 2)
    assert fl3 == sum(3.0 * (m - j) + 4.0 * (m - j) * (n - j - 1) for j in range(2, n, 7))
    assert abs(fl - (2.0 * m * n * n - 2.0 / 3.0 * n ** 3)) < 0.02 * fl


def test_tools_and_entry_scripts_compile():
    """Every helper script shipped in the repo at least parses (they only run on a GPU box)."""
    import glob, os, py_compile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = glob.glob(os.path.join(root, "tools", "*.py")) + [os.path.join(root, f) for f in ("bench.py", "__graft_entry__.py", "dhqr_b200.py")]
    assert len(files) > 5
    for f in files:
        py_compile.compile(f, doraise=True)


def test_balanced_splits_follow_the_reference_formulas():
    # T:35: round((N / sqrt(np)) * sqrt(p))   and   T:36: round(N * (1 - sqrt((np - p) / np)))
    for P, n in ((2, 4096), (4, 4096), (8, 8192), (3, 100), (4, 3)):
        for rule, f in (("trailing", lambda p: n * (p / P) ** 0.5), ("upstream", lambda p: n * (1 - ((P - p) / P) ** 0.5))):
            b = D.balanced_splits(P, n, rule)
            assert len(b) == P + 1 and b[0] == 0 and b[-1] == n and all(b[i] <= b[i + 1] for i in range(P))
            for p in range(1, P):
                assert b[p] == max(b[p - 1], int(round(f(p))))
    assert D.balanced_splits(2, 4096, "upstream") == [0, 1200, 4096]
    assert D.balanced_splits(2, 4096) == [0, 2896, 4096]
    with pytest.raises(ValueError):
        D.balanced_splits(2, 10, "nope")
    # trailing-update work of the right-looking factorisation per rank: reflector j (length m - j) touches the local columns
    # right of j.  The T:35 split evens it out compared with the default distribution; the T:36 split does the opposite.
    m, n, P = 32768, 4096, 4

    def work(bounds):
        j = np.arange(n)
        return np.array([float(np.sum((m - j) * np.clip(bounds[p + 1] - np.maximum(j + 1, bounds[p]), 0, None))) for p in range(P)])

    imb = lambda w: w.max() / w.mean()
    assert imb(work(D.balanced_splits(P, n))) < 1.1 < imb(work(D.splits(P, n))) < imb(work(D.balanced_splits(P, n, "upstream")))


def test_bench_dump_columns_are_fixed_and_within_budget():
    """--dump-outputs writes the same seeded column sample of the factored A on every run with the same shape, at most
    48 MiB of it, and assembles it from DArray-style column blocks exactly as from the whole matrix."""
    import os, sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    assert np.array_equal(bench.dump_columns(2048, 256), np.arange(256))
    cols = bench.dump_columns(32768, 4096)
    assert np.array_equal(cols, bench.dump_columns(32768, 4096)) and 32768 * len(cols) * 8 <= bench.DUMP_A_BYTES
    assert len(set(cols.tolist())) == len(cols) and np.all(np.diff(cols) > 0) and cols[-1] < 4096
    m, n = 9000, 1000
    H = D.colmajor_empty(m, n, device="cpu")
    H.copy_(torch.rand(m, n, dtype=torch.float64))
    alpha = torch.rand(n, dtype=torch.float64)
    whole = bench.gather_outputs(torch, None, H, alpha, m, n, 0, n, 1, "cpu")
    sel = bench.dump_columns(m, n)
    assert len(sel) < n and np.array_equal(whole["A"], H.numpy()[:, sel]) and np.array_equal(whole["alpha"], alpha.numpy())
    b = D.splits(3, n)
    parts = [bench.gather_outputs(torch, None, H[:, b[r]:b[r + 1]], alpha, m, n, b[r], b[r + 1] - b[r], 1, "cpu")["A"] for r in range(3)]
    assert np.array_equal(sum(parts), whole["A"])
