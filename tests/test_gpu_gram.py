"""K2 inside the engine: G / Xty after appends, compactions and the build-ahead layout against numpy (rtol 1e-12).
The kernels themselves are compared with exact and long-double references in tests/test_gpu_gram_ref.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_engine_gram_state_append_and_compact(engine, phis_cubic):
    """Engine-level: G, Xty after appends and a compaction equal numpy on the oracle's X."""
    import fokl_oracle as fo
    rng = np.random.default_rng(11)
    n, m = 3000, 3
    x = rng.random((n, m))
    y = rng.standard_normal(n)
    engine.set_phis(phis_cubic, fo.CUBIC)
    ds = engine.upload(x, y)
    engine.begin_fit(ds)
    t1 = fo.distinct_perms([1, 0, 0]).astype(int)
    t2 = fo.distinct_perms([1, 1, 0]).astype(int)
    engine.append_terms(t1)
    engine.append_terms(t2)
    terms = np.vstack([t1, t2])
    Xh = np.hstack([np.ones((n, 1)), fo.basis_columns(x, terms, phis_cubic, fo.CUBIC)])
    P = engine.P
    assert P == Xh.shape[1]
    G = engine.G[:P, :P].cpu().numpy()
    Xty = engine.Xty[:P].cpu().numpy()
    assert np.allclose(G, Xh.T @ Xh, rtol=1e-12, atol=1e-9)
    assert np.allclose(Xty, Xh.T @ y, rtol=1e-10, atol=1e-9)
    assert np.array_equal(G, G.T)
    assert abs(engine.sum_y - y.sum()) < 1e-9 and abs(engine.yty - y @ y) < 1e-9 and engine.n_global == n
    keep = [0, 1, 3, 4, 6]
    engine.compact(keep)
    G2 = engine.G[:5, :5].cpu().numpy()
    assert np.array_equal(G2, G[np.ix_(keep, keep)])
    assert np.array_equal(engine.Xty[:5].cpu().numpy(), Xty[keep])
    Xd = engine.X[:5, :n].t().cpu().numpy()
    assert np.array_equal(Xd, Xh[:, keep])


def test_engine_build_ahead_layout(engine, phis_cubic):
    """Engine-level: a block started ahead of time above a gap, committed after a compaction, with the cross block
    against the survivors: G / Xty equal numpy and equal the synchronous two-part build bit for bit; residual pass and
    later compactions see the right physical columns."""
    import fokl_oracle as fo
    rng = np.random.default_rng(12)
    n, m = 5000, 3
    x = rng.random((n, m))
    y = rng.standard_normal(n)
    engine.set_phis(phis_cubic, fo.CUBIC)
    ds = engine.upload(x, y)
    t1 = fo.distinct_perms([1, 0, 0]).astype(int)
    t2 = fo.distinct_perms([1, 1, 0]).astype(int)
    t3 = fo.distinct_perms([2, 1, 0]).astype(int)
    t4 = fo.distinct_perms([1, 1, 1]).astype(int)
    results = []
    for ahead in (True, False):
        engine.begin_fit(ds)
        engine.append_terms(t1)                        # P = 4
        p0 = engine.P
        engine.append_terms(t2, p_stable=p0)           # P = 7, synchronous two-part build
        if ahead:
            assert engine.prefetch_terms(t3, p0) is not None      # columns 0 .. 3 are final whatever happens to t2
        keep = [0, 1, 2, 3, 5]                         # t2 loses two columns
        engine.compact(keep)
        p1 = engine.P
        engine.append_terms(t3, p_stable=p0)           # commits the block built ahead (or builds it now)
        if ahead:
            assert engine.gap > 0
            assert engine.prefetch_terms(t4, p1) is not None
        keep2 = list(range(p1)) + [p1 + 1, p1 + 4]
        cols = np.array(keep2, dtype=np.int32)
        bh = engine.evaluate([keep2], engine.make_hypers(4, 1, 4, 1, 1, 1, 10), refine_tol=None).betahat
        ev_res = engine.residual_bic(cols, bh[:len(keep2)])
        engine.compact(keep2)
        engine.append_terms(t4, p_stable=p1)
        P = engine.P
        results.append((engine.G[:P, :P].cpu().numpy(), engine.Xty[:P].cpu().numpy(),
                        engine.X[:P, :n].t().cpu().numpy() if engine.gap == 0 else
                        engine.X[torch_idx(engine, P), :n].t().cpu().numpy(), ev_res))
    terms = np.vstack([t1, t2[[1]], t3[[1, 4]], t4])
    Xh = np.hstack([np.ones((n, 1)), fo.basis_columns(x, terms, phis_cubic, fo.CUBIC)])
    for G, Xty, Xd, _ in results:
        assert np.array_equal(Xd, Xh)
        assert np.allclose(G, Xh.T @ Xh, rtol=1e-12, atol=1e-9) and np.array_equal(G, G.T)
        assert np.allclose(Xty, Xh.T @ y, rtol=1e-10, atol=1e-9)
    assert np.array_equal(results[0][0], results[1][0]) and np.array_equal(results[0][1], results[1][1])
    assert results[0][3] == results[1][3]
    engine.drop_prefetch()


def torch_idx(engine, P):
    import torch
    return torch.as_tensor(engine.phys_cols(np.arange(P)).astype(np.int64), device=engine.device)
