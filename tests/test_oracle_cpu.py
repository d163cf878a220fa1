"""CPU tests: the oracle against the golden fixtures and its own internal consistency."""
import os
import tempfile

import numpy as np

from disn_b200 import synth
from oracle import disn_oracle as orc


def test_chunking_matches_reference_expressions(golden):
    for sdf_res, R, total, split, nsp in golden["chunking"]["table"]:
        assert orc.chunking(int(sdf_res)) == (R, total, split, nsp)
    # SURVEY.md 8: known answers of the driver arithmetic
    assert orc.chunking(64) == (65, 274625, 2, 137313)
    assert orc.chunking(128) == (129, 2146689, 10, 214669)
    assert orc.chunking(256) == (257, 16974593, 80, 212183)
    assert orc.chunking(512) == (513, 135005697, 629, 214636)


def test_cameras_match_reference_preprocessing(golden):
    cam = golden["cameras"]
    for p, ref in zip(cam["params"], cam["trans_mat"]):
        mine = synth.make_trans_mat(p[0], p[1], p[2], p[3], p[4:7])
        np.testing.assert_allclose(mine, ref, rtol=0, atol=2e-5)
    np.testing.assert_allclose(synth.intrinsics(), cam["K"][0], atol=0)
    # cam_est/model_cam.py:28
    np.testing.assert_array_equal(synth.intrinsics(), [[149.84375, 0, 68.5], [0, 149.84375, 68.5], [0, 0, 1]])
    # demo constant reproduced from the commented cam_gt (SURVEY.md 4, item 4)
    assert np.abs(cam["trans_mat"][0] - synth.DEMO_TRANS_MAT[0]).max() < 1e-5


def test_dist_writer_matches_reference_reader(golden):
    g = golden["dist_roundtrip"]
    res = int(g["res"])
    with tempfile.TemporaryDirectory() as td:
        fn = os.path.join(td, "o.dist")
        orc.to_binary(res, list(g["bbox"]), g["values"].astype(np.float64), fn)
        assert np.array_equal(np.fromfile(fn, dtype=np.uint8), g["file_bytes"])


def test_oracle_regression_pin(golden, he_weights):
    g = golden["oracle_small"]
    imgs = synth.synthetic_images(1)
    out = orc.get_model(imgs, g["pts"], g["pts"], synth.DEMO_TRANS_MAT, he_weights, dtype=np.float32)
    np.testing.assert_allclose(out["pred_sdf"], g["pred32"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(out["sample_img_points"], g["uv"], rtol=0, atol=1e-4)
    np.testing.assert_allclose(out["img_embedding"], g["emb32"], rtol=1e-4, atol=1e-5)
    # the synthetic He-scaled weights give O(1) predictions, so a 1e-4 bar on pred/10 is not vacuous
    assert 0.3 < float(np.sqrt(np.mean(g["pred64"] ** 2))) < 3.0
    assert np.abs(g["pred32"] - g["pred64"]).max() < 1e-4


def test_folded_formulation_equals_graph(he_weights):
    """The two algebraic folds the CUDA path uses are exact (checked in float64)."""
    imgs = synth.synthetic_images(1, seed=77)
    pts = np.random.default_rng(3).uniform(-1, 1, size=(1, 256, 3)).astype(np.float32)
    tm = synth.synthetic_trans_mats(1)
    enc = orc.encode(imgs, he_weights, dtype=np.float64)
    ref = orc.decode(enc, pts, pts, tm, he_weights, dtype=np.float64)["pred_sdf"]
    fold = orc.folded_decode(enc, pts, tm, he_weights, dtype=np.float64)
    assert np.abs(ref - fold).max() < 1e-9


def test_tf_resize_semantics():
    # legacy (no half-pixel) bilinear: out[i] samples in[i*scale]; last rows replicate the edge
    x = np.arange(4, dtype=np.float32).reshape(1, 1, 4, 1)
    y = orc.tf_resize_bilinear(x, 1, 8)[0, 0, :, 0]
    np.testing.assert_allclose(y, [0, 0.5, 1, 1.5, 2, 2.5, 3, 3])
    # identity when sizes match
    r = np.random.default_rng(0).random((2, 5, 7, 3), dtype=np.float32)
    np.testing.assert_array_equal(orc.tf_resize_bilinear(r, 5, 7), r)


def test_resampler_semantics():
    data = np.arange(12, dtype=np.float32).reshape(1, 3, 4, 1)     # H=3, W=4
    warp = np.array([[[0, 0], [1.5, 0.5], [3, 2], [3.5, 2], [-0.5, 0], [4.0, 1.0], [-1.0, 0.0]]], np.float32)
    out = orc.tf_resampler(data, warp)[0, :, 0]
    # (3.5,2): right taps fall outside -> contribute 0; (-0.5,0): left taps outside
    np.testing.assert_allclose(out, [0, 3.5, 11, 5.5, 0, 0, 0])


def test_grid_points_order_and_padding():
    pts = orc.grid_points([-1, -1, -1, 1, 1, 1], 3)
    assert pts.shape == (27, 3) and pts.dtype == np.float32
    np.testing.assert_array_equal(pts[0], [-1, -1, -1])
    np.testing.assert_array_equal(pts[1], [0, -1, -1])      # x fastest
    np.testing.assert_array_equal(pts[3], [-1, 0, -1])
    np.testing.assert_array_equal(pts[9], [-1, -1, 0])      # z slowest


def test_get_loss_metrics():
    pred = np.array([[[1.0], [-2.0], [0.5]]], np.float32)
    gt = np.array([[[0.1], [-0.1], [-0.05]]], np.float32)
    m = orc.get_loss(pred, gt)
    assert abs(m["accuracy"] - 2 / 3) < 1e-6
    assert abs(m["sdf_loss_realvalue"] - np.mean([0.0, 0.1, 0.1])) < 1e-6


def test_nn_distance_oracle_matches_reference_compiled_op(golden):
    """oracle/metrics_oracle.nn_distance == the reference's own CPU op compiled in place (oracle/_ref), through its outputs
    at these inputs stored by tests/golden/make_golden_ref_calls.py."""
    from oracle import metrics_oracle as mo
    g = golden["ref_op_outputs"]
    rng = np.random.default_rng(0)
    a = rng.standard_normal((3, 257, 3)).astype(np.float32)
    b = rng.standard_normal((3, 100, 3)).astype(np.float32)
    b[1, 5] = b[1, 9]                       # exact tie: the first minimum must win
    ref = [g["cpu_nn_" + k] for k in ("dist1", "idx1", "dist2", "idx2")]
    got = mo.nn_distance(a, b)
    for g, r in zip(got, ref):
        np.testing.assert_array_equal(g, r)
    # 5x6 points, seed 0: the reference's own eyeball check (tf_nndistance_cpu.py:26-48 verify_nn_distance_cup)
    np.random.seed(0)
    x1 = np.random.randn(1, 5, 3).astype(np.float32)
    x2 = np.random.randn(1, 6, 3).astype(np.float32)
    d1, i1, d2, i2 = mo.nn_distance(x1, x2)
    brute = ((x1[0][:, None] - x2[0][None]) ** 2).sum(-1)
    np.testing.assert_allclose(d1[0], brute.min(1), rtol=1e-6)
    np.testing.assert_array_equal(i1[0], brute.argmin(1))


def _approxmatch_golden():
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "approxmatch_ref.npz"))
    return g, sorted({k.rsplit("_", 1)[0] for k in g.files})


def test_approx_match_oracle_matches_reference_compiled_op(golden):
    """oracle/metrics_oracle.approx_match / match_cost == the reference's own CPU ops compiled in place (oracle/_ref), through
    their outputs at these inputs stored by tests/golden/make_golden_ref_calls.py: equal but for the float64 summation order and
    the last bit of expf (measured <= 4e-9 absolute on `match`; the bar is 2 ulp of float32 at 1.0, since numpy's exp differs in
    the last bit between SIMD code paths)."""
    from oracle import metrics_oracle as mo
    g = golden["ref_op_outputs"]
    rng = np.random.default_rng(3)
    for i, (B, N, M) in enumerate(((2, 64, 64), (1, 96, 32), (1, 40, 100), (1, 7, 1))):
        a = rng.uniform(-0.5, 0.5, (B, N, 3)).astype(np.float32)
        b = rng.uniform(-0.5, 0.5, (B, M, 3)).astype(np.float32)
        ref = g["cpu_am%d_match" % i]
        got = mo.approx_match(a, b)
        np.testing.assert_allclose(got, ref, rtol=2.5e-7, atol=2.5e-7)
        np.testing.assert_allclose(mo.match_cost(a, b, ref), g["cpu_am%d_cost" % i], rtol=1e-7)
        # what a point can give / take bounds its row / column mass (tf_approxmatch.cpp:25-27)
        assert (got.sum(axis=2) <= max(N, M) // N + 1e-5).all() and (got.sum(axis=1) <= max(N, M) // M + 1e-5).all()


def test_approx_match_oracle_against_golden_reference_outputs():
    """The committed outputs of the reference's CPU ops (tests/golden/make_golden_approxmatch.py) -- runs where
    /root/reference and oracle/_ref do not exist."""
    from oracle import metrics_oracle as mo
    g, names = _approxmatch_golden()
    assert names == ["dups", "same", "single", "square", "tall", "wide"]
    for n in names:
        a, b = g[n + "_xyz1"], g[n + "_xyz2"]
        m = mo.approx_match(a, b)
        np.testing.assert_allclose(m, g[n + "_match"], rtol=2.5e-7, atol=2.5e-7, err_msg=n)
        np.testing.assert_allclose(mo.match_cost(a, b, g[n + "_match"]), g[n + "_cost"], rtol=1e-7, atol=1e-12, err_msg=n)
    # identical clouds: everything stays in place, the distance is ~0 (4e-9 from the 1e-9 regularisers)
    assert g["same_cost"][0] < 1e-6
    assert np.allclose(np.diagonal(g["same_match"][0]), 1.0, atol=1e-6)
    # test/test_cd_emd.py:308
    np.testing.assert_allclose(mo.emd(g["square_xyz1"], g["square_xyz2"]), g["square_cost"] * np.float32(0.01), rtol=1e-6)


def test_rotation_from_ortho6d_is_orthonormal_and_right_handed():
    """models/posenet.py:22-36: columns (x, y, z) orthonormal with z = x × y_raw normalised, det +1."""
    from oracle import disn_oracle as orc
    rng = np.random.default_rng(0)
    R = orc.rotation_from_ortho6d(rng.standard_normal((16, 6)))
    np.testing.assert_allclose(np.einsum("bij,bik->bjk", R, R), np.broadcast_to(np.eye(3), (16, 3, 3)), atol=1e-12)
    np.testing.assert_allclose(np.linalg.det(R), 1.0, atol=1e-12)
    # already-orthonormal input is reproduced
    eye6 = np.array([[1., 0, 0, 0, 1, 0]])
    np.testing.assert_allclose(orc.rotation_from_ortho6d(eye6)[0], np.eye(3), atol=0)


def test_nn_distance_oracle_matches_reference_golden(golden):
    """tests/golden/nn_distance_ref.npz holds outputs of the reference's own CPU op (tf_nndistance.cpp compiled in place)."""
    from oracle import metrics_oracle as mo
    g = golden["nn_distance_ref"]
    for name in ("rand", "single", "lattice"):
        got = mo.nn_distance(g[name + "_xyz1"], g[name + "_xyz2"])
        for arr, key in zip(got, ("_dist1", "_idx1", "_dist2", "_idx2")):
            np.testing.assert_array_equal(arr, g[name + key], err_msg=name + key)


def test_iou_oracle_properties():
    """oracle/metrics_oracle.iou_voxel (restated test/test_iou.py:208-233): identity, disjointness, monotone overlap."""
    from oracle import metrics_oracle as mo

    def box(lo, hi):
        lo, hi = np.asarray(lo, np.float32), np.asarray(hi, np.float32)
        v = np.array([[x, y, z] for z in (lo[2], hi[2]) for y in (lo[1], hi[1]) for x in (lo[0], hi[0])], np.float32)
        f = np.array([[0, 1, 3], [0, 3, 2], [4, 6, 7], [4, 7, 5], [0, 4, 5], [0, 5, 1], [2, 3, 7], [2, 7, 6],
                      [0, 2, 6], [0, 6, 4], [1, 5, 7], [1, 7, 3]], np.int32)
        return v, f
    a = box((-0.3, -0.3, -0.3), (0.3, 0.3, 0.3))
    b = box((-0.3, -0.3, -0.3), (0.3, 0.3, 0.1))
    c = box((0.6, 0.6, 0.6), (0.8, 0.8, 0.8))
    assert mo.iou_voxel(*a, *a, dim=32)[2] == 1.0
    assert mo.iou_voxel(*a, *c, dim=32)[2] == 0.0
    i_ab = mo.iou_voxel(*a, *b, dim=32)[2]
    assert 0.3 < i_ab < 1.0
    occ = mo.voxel_occupancy(*a, dim=32)
    assert occ.sum() > 0 and occ[0, 0, 0] == 0          # surface voxels only, binned inside the grid
    # the surface of the box is hollow in the occupancy grid: the centre bin is empty
    ctr = int((0.0 + 1.1) / 2.4 * 32)
    assert occ[ctr, ctr, ctr] == 0
