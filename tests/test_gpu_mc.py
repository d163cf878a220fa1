"""GPU tests of the CUDA marching-cubes post-pass against the CPU oracle (bit-exact integer topology)."""
import numpy as np
import pytest

from oracle import mc_oracle as mco

pytestmark = pytest.mark.gpu


def _sphere(R, r=0.6, c=(0.05, -0.1, 0.02)):
    ax = np.linspace(-1, 1, R)
    z, y, x = np.meshgrid(ax, ax, ax, indexing="ij")
    return (np.sqrt((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2) - r).astype(np.float32)


@pytest.mark.parametrize("case", ["sphere33", "sphere65_iso", "random17", "random40", "empty", "nonuniform_box"])
def test_marching_cubes_matches_oracle_bit_exact(engine, case):
    bbox = [-1, -1, -1, 1, 1, 1]
    iso = 0.0
    if case == "sphere33":
        sdf = _sphere(33)
    elif case == "sphere65_iso":
        sdf, iso = _sphere(65), 0.0371
    elif case in ("random17", "random40"):
        R = int(case[6:])
        sdf = np.random.default_rng(R).standard_normal((R, R, R)).astype(np.float32)   # every ambiguous case
    elif case == "empty":
        sdf = np.ones((9, 9, 9), np.float32)
    else:
        sdf, bbox = _sphere(21), [-1.0, -0.9, -0.8, 1.0, 0.7, 0.9]
    v, f = engine.marching_cubes(sdf, bbox, iso)
    rv, rf = mco.marching_cubes(sdf, bbox, iso)
    assert v.shape == rv.shape and f.shape == rf.shape
    np.testing.assert_array_equal(f, rf)            # integer topology: bit-exact
    np.testing.assert_array_equal(v, rv)            # same float64 formula, same roundings
    if case.startswith("sphere"):
        assert mco.is_closed_manifold(f) and mco.signed_volume(v, f) > 0     # outward winding like demo/result.obj


def test_mesh_of_predicted_grid_is_consistent(engine, he_weights):
    """SDF grid -> CUDA marching cubes at iso = median (synthetic fields need not cross zero)."""
    from disn_b200 import synth
    engine.encode(synth.synthetic_images(1))
    grid = engine.eval_grid(synth.DEMO_SDF_PARAMS, synth.DEMO_TRANS_MAT, 24)[0]
    iso = float(np.median(grid))
    v, f = engine.marching_cubes(grid, [-1, -1, -1, 1, 1, 1], iso)
    rv, rf = mco.marching_cubes(grid, [-1, -1, -1, 1, 1, 1], iso)
    assert len(f) > 100
    np.testing.assert_array_equal(f, rf)
    np.testing.assert_array_equal(v, rv)


def test_nn_distance_bit_exact_vs_reference_op(engine, golden):
    """CUDA NnDistance == the CPU oracle == the reference's own compiled op (its outputs at these inputs, stored by
    tests/golden/make_golden_ref_calls.py): shapes of the reference call site (test/test_cd_emd.py:42-45: [views,2048,3])."""
    from oracle import metrics_oracle as mo
    rng = np.random.default_rng(7)
    a = rng.uniform(-1, 1, (4, 2048, 3)).astype(np.float32)
    b = rng.uniform(-1, 1, (4, 1500, 3)).astype(np.float32)
    b[2, 10] = b[2, 700]                                    # exact tie -> first index wins
    got = engine.nn_distance(a, b)
    ref = mo.nn_distance(a, b)
    for g, r in zip(got, ref):
        np.testing.assert_array_equal(g, r)
    for g, key in zip(got, ("dist1", "idx1", "dist2", "idx2")):
        np.testing.assert_array_equal(g, golden["ref_op_outputs"]["gpu_nn_" + key], err_msg=key)
    np.testing.assert_allclose(engine.chamfer_x1000(a, b), mo.chamfer_x1000(a, b), rtol=1e-6)
    th = [0.005, 0.01, 0.02, 0.05, 0.1]
    for got, want in zip(engine.f_score(a[:1], b[:1], th), mo.precision_recall_f(a[:1], b[:1], th)):
        np.testing.assert_array_equal(got, want)        # distances are bit-identical, so the counts are
    from disn_b200._lib import DisnError
    with pytest.raises(DisnError):
        engine.nn_distance(a[:, :0], b)                     # empty set: loud error like the op's shape checks


def test_nn_distance_matches_reference_golden(engine, golden):
    """CUDA kernel vs outputs of the reference's own CPU op (committed fixture; the GPU box has no /root/reference)."""
    g = golden["nn_distance_ref"]
    for name in ("rand", "single", "lattice"):
        got = engine.nn_distance(g[name + "_xyz1"], g[name + "_xyz2"])
        for arr, key in zip(got, ("_dist1", "_idx1", "_dist2", "_idx2")):
            np.testing.assert_array_equal(arr, g[name + key], err_msg=name + key)
