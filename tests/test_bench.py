"""bench.py's output dump (names, dtypes, the size cap and its fixed row sample), its argument checks, and the
fixed-point member sums that make the benchmark's index training reproducible."""
import os
import sys

import numpy as np
import pytest
import torch

import bench


class HostAssign:
    """Host stand-in for the assignment kernels of train.LibrsbOps."""

    def assign_ip(self, x, c):
        return (x @ c.T).argmax(1)

    def pq_assign(self, r, cb):
        M, _, dsub = cb.shape
        return torch.cdist(r.reshape(-1, M, dsub).permute(1, 0, 2), cb).argmin(2).T.contiguous().to(torch.uint8)


def test_fixed_point_sums_are_exact_and_independent_of_row_order():
    g = torch.Generator().manual_seed(0)
    n, d, k = 5000, 24, 40
    x = torch.randn(n, d, generator=g) * torch.logspace(-4, 1, d)          # columns of very different magnitude
    seg = torch.randint(0, k - 3, (n,), generator=g)                          # the last 3 segments stay empty
    s = bench.fixed_point_sums(x, seg, k, chunk_elems=777 * d)
    perm = torch.randperm(n, generator=g)
    assert torch.equal(s, bench.fixed_point_sums(x[perm], seg[perm], k, chunk_elems=1000 * d))
    exact = torch.zeros(k, d, dtype=torch.float64).index_add_(0, seg, x.double())
    assert torch.allclose(s.double(), exact, rtol=2e-7, atol=1e-10)
    assert not s[k - 3:].any()
    assert not bench.fixed_point_sums(torch.zeros(4, 3), torch.zeros(4, dtype=torch.int64), 2).any()


def test_reproducible_training_ops_sum_what_the_definition_sums():
    g = torch.Generator().manual_seed(1)
    ops = bench.ReproducibleTrainingOps(HostAssign())
    x = torch.randn(3000, 32, generator=g)
    a = ops.assign_ip(x, torch.randn(20, 32, generator=g))
    sums, counts = ops.accumulate(x, a, 20)
    assert torch.equal(counts, torch.bincount(a, minlength=20).float())
    assert torch.allclose(sums, torch.zeros(20, 32).index_add_(0, a, x), rtol=1e-5, atol=1e-5)
    M, ksub = 8, 256
    codes = ops.pq_assign(x, torch.randn(M, ksub, 32 // M, generator=g))
    sums, counts = ops.pq_accumulate(x, codes, M, ksub)
    xm = x.reshape(-1, M, 32 // M)
    for m in range(M):
        c = codes[:, m].long()
        assert torch.equal(counts[m], torch.bincount(c, minlength=ksub).float())
        assert torch.allclose(sums[m], torch.zeros(ksub, 32 // M).index_add_(0, c, xm[:, m]), rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
def test_reproducible_training_matches_librsb_kernels_and_repeats_exactly():
    from retrieval_scaling_b200 import train
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(20000, 128, generator=g, device="cuda")
    lib_ops = train.LibrsbOps()
    ops = bench.ReproducibleTrainingOps(lib_ops)
    a = ops.assign_ip(x, torch.nn.functional.normalize(torch.randn(32, 128, generator=g, device="cuda"), dim=1))
    (s, c), (s0, c0) = ops.accumulate(x, a, 32), lib_ops.accumulate(x, a, 32)
    assert torch.equal(c, c0) and torch.allclose(s, s0, rtol=1e-5, atol=1e-3)
    codes = ops.pq_assign(x, torch.randn(16, 256, 8, generator=g, device="cuda"))
    (s, c), (s0, c0) = ops.pq_accumulate(x, codes, 16, 256), lib_ops.pq_accumulate(x, codes, 16, 256)
    assert torch.equal(c, c0) and torch.allclose(s, s0, rtol=1e-5, atol=1e-3)
    runs = [train.kmeans(x, 32, niter=5, spherical=True, seed=3, ops=bench.ReproducibleTrainingOps(train.LibrsbOps()))
            for _ in range(2)]
    assert torch.equal(runs[0], runs[1])
    cbs = [train.train_pq(x, 16, 256, niter=5, seed=3, ops=bench.ReproducibleTrainingOps(train.LibrsbOps())) for _ in range(2)]
    assert torch.equal(cbs[0], cbs[1])


def test_dump_writes_ids_and_scores(tmp_path):
    I = torch.arange(60, dtype=torch.int64).reshape(6, 10) + (1 << 40)      # ids past 2**32 stay exact in float64
    I[5, 7:] = -1                                                            # padding of a short result row
    D = torch.linspace(-1.0, 1.0, 60).reshape(6, 10)
    assert bench.dump_outputs(str(tmp_path / "d"), I, D) == {"ids": [6, 10], "scores": [6, 10]}
    ids, scores = np.load(tmp_path / "d" / "ids.npy"), np.load(tmp_path / "d" / "scores.npy")
    assert ids.dtype == np.float64 and scores.dtype == np.float32
    assert np.array_equal(ids.astype(np.int64), I.numpy()) and np.array_equal(scores, D.numpy())
    assert sorted(os.listdir(tmp_path / "d")) == ["ids.npy", "scores.npy"]


def test_dump_above_the_limit_writes_a_fixed_sample_of_rows(tmp_path):
    nq, k, keep = 1000, 10, 100
    I = torch.arange(nq * k, dtype=torch.int64).reshape(nq, k)
    D = torch.randn(nq, k)
    limit = 4096 + keep * (k * 12 + 8)
    for run in ("a", "b"):
        assert bench.dump_outputs(str(tmp_path / run), I, D, limit=limit) == \
            {"ids": [keep, k], "scores": [keep, k], "rows": [keep]}
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= limit
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    r = rows.astype(np.int64)
    assert np.array_equal(r, np.unique(r)) and r[0] >= 0 and r[-1] < nq
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy").astype(np.int64), I.numpy()[r])
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), D.numpy()[r])


def test_steps_and_warmup_are_parsed(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "7", "--warmup", "0", "--dump-outputs", "out"])
    args = bench.parse()
    assert (args.steps, args.warmup, args.dump_outputs) == (7, 0, "out")


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"],
                                  ["--encoder-only", "--dump-outputs", "out"]])
def test_bench_rejects(argv, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.parse()
    assert e.value.code == 2
