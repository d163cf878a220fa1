"""GPU tests of the remaining reference surface: graph intermediates and the encoder/decoder split point
(models/model_normalization.py:38-45,169-206,223-238), the literal chunk loop, the device-resident driver tail, and the
IoU evaluator (test/test_iou.py:208-233)."""
import os

import numpy as np
import pytest

from disn_b200 import synth
from oracle import disn_oracle as orc
from oracle import mc_oracle as mco
from oracle import metrics_oracle as mo

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("precision", ["fp32", "f16f8"])
def test_intermediates_and_decoder_split_point(he_weights, precision):
    from disn_b200 import create_sdf as cs
    from disn_b200 import model_normalization as model
    F = cs.default_flags(sdf_res=8)
    B, N = 2, 257
    pls = model.placeholder_inputs(B, 1, (137, 137), num_sample_pc=N, scope="inputs_pl", FLAGS=F)
    itp = model.Placeholder("is_training", ())
    ep = model.get_model(pls, 1, itp, bn=False, FLAGS=F)
    feat_pls = model.placeholder_features(B, num_sample_pc=N)
    dec = model.get_decoder(N, pls, feat_pls)
    imgs = synth.synthetic_images(B, seed=71)
    rng = np.random.default_rng(72)
    pts = rng.uniform(-1, 1, size=(B, N, 3)).astype(np.float32)
    rot = rng.uniform(-1, 1, size=(B, N, 3)).astype(np.float32)
    tm = np.concatenate([synth.DEMO_TRANS_MAT, synth.synthetic_trans_mats(1, seed=9)], axis=0)
    ref = orc.get_model(imgs, pts, rot, tm, he_weights, dtype=np.float64)
    sess = model.Session(weights=he_weights, precision=precision, max_batch=B)
    try:
        feed = {itp: False, pls["sample_pc"]: pts, pls["sample_pc_rot"]: rot, pls["imgs"]: imgs, pls["trans_mat"]: tm}
        pred, pg, pl_, feat, uv = sess.run([ep["pred_sdf"], ep["pred_sdf_value_global"], ep["pred_sdf_value_local"],
                                            ep["point_img_feat"], ep["sample_img_points"]], feed_dict=feed)
        assert feat.shape == (B, N, 1, 1472)
        np.testing.assert_allclose(uv, ref["sample_img_points"], atol=2e-4)
        fs = float(np.abs(ref["point_img_feat"]).max())
        assert np.abs(feat - ref["point_img_feat"]).max() <= 1e-4 * fs           # taps are bf16x3 / fp32 convs
        for got, key in ((pred, "pred_sdf"), (pg, "pred_sdf_value_global"), (pl_, "pred_sdf_value_local")):
            assert np.abs(got - ref[key]).max() / orc.SDF_WEIGHT <= 1e-4, key
        np.testing.assert_allclose(pg + pl_, pred, atol=1e-6)
        # get_decoder: feed the oracle's own features (float32 like a caller would) and compare with its decode
        emb = ref["img_embedding"].astype(np.float32).reshape(B, 1, 1, 1024)
        pf = ref["point_img_feat"].astype(np.float32)
        out = sess.run(dec, feed_dict={pls["sample_pc_rot"]: rot, feat_pls["ref_feats_embedding_cnn"]: emb,
                                       feat_pls["point_img_feat"]: pf})
        assert out.shape == (B, N, 1)
        assert np.abs(out - ref["pred_sdf"]).max() / orc.SDF_WEIGHT <= 1e-4
        # the two sdfnet heads on their own (models/sdfnet.py:69,171): symbolic through Session.run and eager on arrays
        from disn_b200 import sdfnet
        hp = model.Placeholder("src_pc", (B, N, 3))
        hg = model.Placeholder("globalfeats", (B, 1, 1, 1024))
        hf = model.Placeholder("point_feat", (B, N, 1, 1472))
        tg = sdfnet.get_sdf_basic2(hp, hg, False, B, N, False, None)
        tl = sdfnet.get_sdf_basic2_imgfeat_twostream(hp, hf, False, B, N, False, None)
        og, ol = sess.run([tg, tl], feed_dict={hp: rot, hg: emb, hf: pf})
        assert np.abs(og - ref["pred_sdf_value_global"]).max() / orc.SDF_WEIGHT <= 1e-4
        assert np.abs(ol - ref["pred_sdf_value_local"]).max() / orc.SDF_WEIGHT <= 1e-4
        sdfnet.set_engine(sess.engine)
        np.testing.assert_array_equal(sdfnet.get_sdf_basic2(rot, emb, False, B, N, False, None), og)
        sdfnet.set_engine(None)
        # and our own fetched features close the loop: decoder(point_img_feat, embedding) == fused pred_sdf
        out2 = sess.run(dec, feed_dict={pls["sample_pc_rot"]: rot,
                                        feat_pls["ref_feats_embedding_cnn"]: sess.engine.get_encoded(0).reshape(B, 1, 1, 1024),
                                        feat_pls["point_img_feat"]: feat})
        assert np.abs(out2 - pred).max() / orc.SDF_WEIGHT <= 2e-5
    finally:
        sess.close()


def test_decoder_staging_survives_nn_distance(he_weights):
    """nn_distance grows the context's device staging between decoder calls (eval_points_ex, point_img_feat,
    eval_features): repeating those calls must give the same bits, and a larger one afterwards must match a fresh
    context's."""
    from disn_b200.engine import Engine
    B = 2
    imgs, tm = synth.synthetic_images(B, seed=31), synth.synthetic_trans_mats(B, seed=32)

    def open_engine():
        eng = Engine(device=0, precision="f16f8", max_batch=B)
        eng.load_weights(he_weights)
        eng.encode(imgs)
        return eng

    def decode(eng, N):
        pts = np.random.default_rng(N).uniform(-1, 1, size=(B, N, 3)).astype(np.float32)
        feat, uv = eng.point_img_feat(pts, tm)
        return eng.eval_points_ex(pts, tm) + (feat, uv) + eng.eval_features(pts, eng.get_encoded(0), feat)

    eng = open_engine()
    try:
        small = decode(eng, 64)
        rng = np.random.default_rng(34)
        a, b = (rng.uniform(-1, 1, size=(B, 20000, 3)).astype(np.float32) for _ in range(2))
        d1, i1, d2, i2 = eng.nn_distance(a, b)     # 1.6 MB of staging: more than the decoder calls above needed
        for k in (0, 777, 19999):
            np.testing.assert_allclose(d1[1, k], ((b[1] - a[1, k]) ** 2).sum(-1).min(), rtol=1e-5, atol=1e-7)
            np.testing.assert_allclose(d2[0, k], ((a[0] - b[0, k]) ** 2).sum(-1).min(), rtol=1e-5, atol=1e-7)
        for got, want in zip(decode(eng, 64), small):
            np.testing.assert_array_equal(got, want)
        large = decode(eng, 1500)
    finally:
        eng.close()
    fresh = open_engine()
    try:
        for got, want in zip(large, decode(fresh, 1500)):
            np.testing.assert_array_equal(got, want)
    finally:
        fresh.close()


def test_literal_reference_loop_equals_device_grid(he_weights, tmp_path):
    """create_sdf.py:241-285 replayed literally (tests/reference_loop.py) == one disn_eval_grid call, bit for bit."""
    from disn_b200 import create_sdf as cs
    from disn_b200 import model_normalization as model
    from tests import reference_loop
    F = cs.default_flags(sdf_res=12, log_dir=str(tmp_path / "log"), batch_size=2, precision="f16f8")
    cs.configure(F)
    pls = model.placeholder_inputs(2, 1, (137, 137), num_sample_pc=cs.NUM_SAMPLE_POINTS, FLAGS=F)
    itp = model.Placeholder("is_training", ())
    ep = model.get_model(pls, 1, itp, FLAGS=F)
    ops = {"input_pls": pls, "is_training_pl": itp, "end_points": ep}
    batch = {"img": synth.synthetic_images(2, seed=5), "trans_mat": synth.synthetic_trans_mats(2, seed=6),
             "sdf_params": np.array([[-1, -1, -1, 1, 1, 1], [-0.9, -1, -0.8, 1, 0.7, 0.95]], np.float64)}
    sess = model.Session(weights=he_weights, precision="f16f8", max_batch=2)
    try:
        lit = reference_loop.run_literal(cs, sess, ops, batch)
        grid = sess.engine.eval_grid(batch["sdf_params"], batch["trans_mat"], 12)
        np.testing.assert_array_equal(lit.astype(np.float32).reshape(grid.shape), grid)
    finally:
        sess.close()


def test_driver_keeps_the_grid_on_the_device(he_weights, tmp_path):
    """create(): encode -> resident grid -> CUDA marching cubes on that buffer -> OBJ; the optional .dist artefact is
    byte-identical to the reference writer's and meshes to the same topology on the CPU oracle."""
    from disn_b200 import create_sdf as cs
    F = cs.default_flags(sdf_res=24, log_dir=str(tmp_path / "log"), iso=0.0, batch_size=2, precision="f16f8", keep_dist=True)
    cs.configure(F)
    imgs = synth.synthetic_images(2, seed=41)
    batch = {"img": imgs, "trans_mat": synth.synthetic_trans_mats(2, seed=42),
             "sdf_params": np.tile(synth.DEMO_SDF_PARAMS, (2, 1)), "cat_id": ["02691156", "03001627"],
             "obj_nm": ["a", "b"], "view_id": [0, 23]}
    from disn_b200.engine import Engine
    eng = Engine(device=0, precision="f16f8", max_batch=2)
    try:
        eng.load_weights(he_weights)
        eng.encode(imgs)
        grid = eng.eval_grid(batch["sdf_params"], batch["trans_mat"], 24)
    finally:
        eng.close()
    F.iso = float(np.median(grid))
    cs.configure(F)
    written = cs.create(he_weights, [batch])
    assert [os.path.basename(w) for w in written] == ["02691156_a_00.obj", "03001627_b_23.obj"]
    for b, w in enumerate(written):
        res, bbox, vals = cs.read_dist(w[:-4] + ".dist")
        assert res == 24
        np.testing.assert_array_equal(vals, grid[b])
        ref_file = str(tmp_path / ("ref%d.dist" % b))
        orc.to_binary(24, list(batch["sdf_params"][b]), grid[b].reshape(-1), ref_file)
        assert open(ref_file, "rb").read() == open(w[:-4] + ".dist", "rb").read()
        rv, rf = mco.marching_cubes(grid[b], batch["sdf_params"][b], F.iso)
        faces = np.array([[int(x) - 1 for x in l.split()[1:]] for l in open(w) if l.startswith("f ")], np.int32)
        np.testing.assert_array_equal(faces, rf)


def _icosphere(radius, centre, sub=2):
    t = (1.0 + 5 ** 0.5) / 2
    v = np.array([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                  [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], np.float64)
    f = np.array([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
                  [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
                  [6, 2, 10], [8, 6, 7], [9, 8, 1]], np.int64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    for _ in range(sub):
        cache, nf, vl = {}, [], list(v)

        def mid(a, b):
            k = (min(a, b), max(a, b))
            if k not in cache:
                m = (vl[a] + vl[b]) / 2
                vl.append(m / np.linalg.norm(m))
                cache[k] = len(vl) - 1
            return cache[k]
        for a, b, c in f:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            nf += [[a, ab, ca], [b, bc, ab], [c, ca, bc], [ab, bc, ca]]
        v, f = np.array(vl), np.array(nf)
    return (v * radius + np.asarray(centre)).astype(np.float32), f.astype(np.int32)


@pytest.mark.parametrize("dim", [110, 32])
def test_iou_matches_cpu_twin(dim):
    """GPU voxeliser + binning + counts == oracle/metrics_oracle.iou_voxel (same float64 operations): equal occupancy
    grids, equal counts; sanity: IoU(A,A) = 1, disjoint meshes -> 0, nested spheres in between."""
    from disn_b200.engine import Engine
    a = _icosphere(0.45, (0.05, -0.02, 0.1))
    b = _icosphere(0.40, (0.12, 0.03, 0.02))
    rng = np.random.default_rng(3)
    tri_v = rng.uniform(-0.8, 0.8, size=(90, 3)).astype(np.float32)          # a random triangle soup (large triangles)
    tri_f = np.arange(90, dtype=np.int32).reshape(30, 3)
    far = _icosphere(0.1, (-0.7, -0.7, -0.7))
    eng = Engine(device=0, precision="fp32")
    try:
        for (v1, f1), (v2, f2) in ((a, b), ((tri_v, tri_f), a)):
            iou, inter, uni, o1, o2 = eng.iou(v1, f1, v2, f2, dim=dim, want_grids=True)
            r1, r2 = mo.voxel_occupancy(v1, f1, dim), mo.voxel_occupancy(v2, f2, dim)
            np.testing.assert_array_equal(o1, r1)
            np.testing.assert_array_equal(o2, r2)
            ri, ru, riou = mo.iou_voxel(v1, f1, v2, f2, dim)
            assert (inter, uni) == (ri, ru) and abs(iou - riou) < 1e-12 and 0 < iou < 1
        assert eng.iou(a[0], a[1], a[0], a[1], dim=dim) == 1.0
        assert eng.iou(a[0], a[1], far[0], far[1], dim=dim) == 0.0
    finally:
        eng.close()


def test_pinned_host_outputs_are_written_by_the_kernel(he_weights):
    """Caller-pinned output buffers (cudaHostAlloc / torch pin_memory) take the zero-copy path -- the kernel's epilogue stores
    into them directly -- and must give the same bits as pageable buffers (device scratch + copy)."""
    import torch
    from disn_b200.engine import Engine
    eng = Engine(device=0, precision="f16f8", max_batch=2)
    try:
        eng.load_weights(he_weights)
        eng.encode(synth.synthetic_images(2, seed=9))
        tm = synth.synthetic_trans_mats(2, seed=3)
        sp = np.tile(synth.DEMO_SDF_PARAMS, (2, 1))
        ref = eng.eval_grid(sp, tm, 24)                                   # pageable numpy output
        pinned = torch.empty(ref.shape, dtype=torch.float32).pin_memory()
        pinned.fill_(float("nan"))
        out = eng.eval_grid(sp, tm, 24, out=pinned.numpy())
        assert out.ctypes.data == pinned.data_ptr()
        np.testing.assert_array_equal(pinned.numpy(), ref)
        # a z-slab into the middle of a pinned whole-grid buffer (what each rank does in the multi-GPU host path)
        eng.encode(synth.synthetic_images(1, seed=9))
        whole = eng.eval_grid(sp[:1], tm[:1], 24)
        pinned.fill_(float("nan"))
        eng.eval_grid(sp[:1], tm[:1], 24, z0=5, z1=17, out=pinned.numpy()[0, 5:17].reshape(1, 12, 25, 25))
        np.testing.assert_array_equal(pinned.numpy()[0, 5:17], whole[0, 5:17])
        assert np.isnan(pinned.numpy()[0, :5]).all() and np.isnan(pinned.numpy()[0, 17:]).all()
        eng.encode(synth.synthetic_images(2, seed=9))
        pts = np.random.default_rng(1).uniform(-1, 1, size=(2, 777, 3)).astype(np.float32)
        ref_p, ref_uv = eng.eval_points(pts, tm, want_uv=True)
        import ctypes as C
        from disn_b200._lib import check
        pp = torch.empty((2, 777, 1), dtype=torch.float32).pin_memory()
        puv = torch.empty((2, 777, 2), dtype=torch.float32).pin_memory()
        check(eng.lib.disn_eval_points(eng._h, pts.ctypes.data_as(C.c_void_p), None, np.ascontiguousarray(tm).ctypes.data_as(C.c_void_p),
                                       2, 777, C.c_void_p(pp.data_ptr()), C.c_void_p(puv.data_ptr()), 0))
        np.testing.assert_array_equal(pp.numpy(), ref_p)
        np.testing.assert_array_equal(puv.numpy(), ref_uv)
    finally:
        eng.close()
