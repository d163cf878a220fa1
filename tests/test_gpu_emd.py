"""GPU tests of the approximate-EMD evaluator (csrc/emd.cu) against the CPU oracle and the committed outputs of the
reference's own CPU ops (models/tf_ops/approxmatch/tf_approxmatch.cpp; tests/golden/make_golden_approxmatch.py).

Tolerances: `match` is a float32 accumulation of float64 terms -- the CUDA path and the CPU ops differ by the float64 summation
order and the rare last bit of expf, i.e. by at most an ulp or two of float32 at the entry's size (entries <= capacity, 1..4;
measured 3e-8): the bar is 2.5e-7 absolute + 2.5e-7 relative.
`cost` (a float64 sum of 1e4..4e6 float32 products, stored as float32): 1e-6 relative."""
import numpy as np
import pytest

from oracle import metrics_oracle as mo

pytestmark = pytest.mark.gpu
MATCH_ATOL = 2.5e-7
MATCH_RTOL = 2.5e-7
COST_RTOL = 1e-6


def test_approx_match_matches_reference_golden(engine, golden):
    g = golden["approxmatch_ref"]
    for name in ("square", "wide", "tall", "single", "dups", "same"):
        a, b = g[name + "_xyz1"], g[name + "_xyz2"]
        m, c = engine.approx_match(a, b, cost=True)
        assert m.shape == g[name + "_match"].shape
        np.testing.assert_allclose(m, g[name + "_match"], rtol=MATCH_RTOL, atol=MATCH_ATOL, err_msg=name)
        np.testing.assert_allclose(c, g[name + "_cost"], rtol=COST_RTOL, atol=1e-7, err_msg=name)
        # the MatchCost op on the reference's own match: only the float64 summation order differs
        np.testing.assert_allclose(engine.match_cost(a, b, g[name + "_match"]), g[name + "_cost"], rtol=COST_RTOL, atol=1e-12,
                                   err_msg=name)


def test_emd_at_the_reference_call_shape(engine, golden):
    """test/test_cd_emd.py:42-45,307-308: [views, 2048, 3] clouds; CUDA vs the CPU oracle and vs the reference's compiled op
    (a sample of its match on the first view, stored by tests/golden/make_golden_ref_calls.py: every row's largest entries and
    entries at seeded indices), mass bounds, run-to-run reproducibility, and the cost-only entry (match never leaves HBM)."""
    rng = np.random.default_rng(11)
    a = rng.uniform(-0.5, 0.5, (2, 2048, 3)).astype(np.float32)
    b = (a[:, rng.permutation(2048)] + rng.normal(0, 0.02, (2, 2048, 3))).astype(np.float32)      # a noisy copy, shuffled
    m, c = engine.approx_match(a, b, cost=True)
    want = mo.approx_match(a, b)
    np.testing.assert_allclose(m, want, rtol=MATCH_RTOL, atol=MATCH_ATOL)
    np.testing.assert_allclose(c, mo.match_cost(a, b, want), rtol=COST_RTOL)
    g = golden["ref_op_outputs"]
    np.testing.assert_allclose(np.take_along_axis(m[0], g["gpu_emd_top_idx"].astype(np.int64), 1), g["gpu_emd_top_val"],
                               rtol=MATCH_RTOL, atol=MATCH_ATOL)
    np.testing.assert_allclose(m[0].reshape(-1)[g["gpu_emd_sample_idx"]], g["gpu_emd_sample_val"], rtol=MATCH_RTOL, atol=MATCH_ATOL)
    assert (m >= 0).all() and (m.sum(axis=2) <= 1 + 1e-4).all() and (m.sum(axis=1) <= 1 + 1e-4).all()
    assert m.sum() > 0.999 * 2 * 2048                         # (nearly) all the mass is moved
    np.testing.assert_allclose(engine.emd(a, b), c * np.float32(0.01), rtol=0, atol=0)
    m2, c2 = engine.approx_match(a, b, cost=True)
    np.testing.assert_array_equal(m, m2)                      # fixed reduction order: bit-reproducible
    np.testing.assert_array_equal(c, c2)
    # a noisy copy is much closer than an unrelated cloud
    far = engine.emd(a, rng.uniform(-0.5, 0.5, (2, 2048, 3)).astype(np.float32))
    assert (engine.emd(a, b) < 0.5 * far).all()


def test_approx_match_ragged_and_errors(engine):
    """N != M (capacity factors max(N,M)/N and max(N,M)/M, integer division as in the op) and the op's shape checks."""
    from disn_b200._lib import DisnError
    rng = np.random.default_rng(12)
    for N, M in ((300, 77), (50, 333), (1, 64)):
        a = rng.uniform(-0.5, 0.5, (3, N, 3)).astype(np.float32)
        b = rng.uniform(-0.5, 0.5, (3, M, 3)).astype(np.float32)
        m, c = engine.approx_match(a, b, cost=True)
        want = mo.approx_match(a, b)
        np.testing.assert_allclose(m, want, rtol=MATCH_RTOL, atol=MATCH_ATOL)
        np.testing.assert_allclose(c, mo.match_cost(a, b, want), rtol=COST_RTOL)
        assert (m.sum(axis=2) <= max(N, M) // N + 1e-4).all() and (m.sum(axis=1) <= max(N, M) // M + 1e-4).all()
    with pytest.raises(DisnError):
        engine.approx_match(a[:, :0], b)
    with pytest.raises(DisnError):
        engine.match_cost(a, b[:, :0], np.zeros((3, 1, 0), np.float32))


def test_points_loss_like_the_evaluation_script(engine):
    """Engine.points_loss == get_points_loss (test/test_cd_emd.py:291-315) evaluated with the CPU oracles."""
    rng = np.random.default_rng(13)
    gt = rng.uniform(-0.5, 0.5, (1, 512, 3)).astype(np.float32)
    views = np.concatenate([gt + rng.normal(0, s, gt.shape).astype(np.float32) for s in (0.05, 0.01, 0.1)], 0)
    got = engine.points_loss(np.concatenate([gt, views], 0))
    src = np.repeat(gt, 3, 0)
    cf, em = mo.chamfer_x1000(views, src), mo.emd(src, views)
    want = (cf.mean(), cf.min(), int(cf.argmin()), em.mean(), em.min(), int(em.argmin()))
    assert got[2] == want[2] == 1 and got[5] == want[5] == 1           # the least noisy view wins both
    np.testing.assert_allclose([got[0], got[1]], [want[0], want[1]], rtol=1e-6)
    np.testing.assert_allclose([got[3], got[4]], [want[3], want[4]], rtol=2e-6)
