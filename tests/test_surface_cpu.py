"""CPU tests of the reference-compatible Python surface, host-only C-ABI entry points and the multi-rank
slab logic (gloo, world_size 2)."""
import os
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest


def _flags(**kw):
    from disn_b200 import create_sdf as cs
    return cs.default_flags(**kw)


def test_placeholders_and_end_points_keys_match_reference():
    from disn_b200 import model_normalization as model
    F = _flags()
    pls = model.placeholder_inputs(2, 1, (137, 137), num_sample_pc=100, scope="inputs_pl", FLAGS=F)
    # models/model_normalization.py:27-35
    assert set(pls) == {"pc", "sample_pc", "sample_pc_rot", "imgs", "sdf", "sdf_params", "trans_mat"}
    assert pls["imgs"].shape == (2, 137, 137, 3) and pls["trans_mat"].shape == (2, 4, 3)
    assert pls["sample_pc"].shape == (2, 100, 3) and pls["sdf"].shape == (2, 100, 1)
    ep = model.get_model(pls, 1, model.Placeholder("is_training", ()), bn=False, FLAGS=F)
    # models/model_normalization.py:60-63,73,79,205-219
    for k in ("ref_pc", "ref_sdf", "ref_img", "resized_ref_img", "img_embedding", "pred_sdf_value_global",
              "pred_sdf_value_local", "pred_sdf", "sample_img_points", "ref_feats_embedding_cnn", "point_img_feat"):
        assert k in ep, k
    loss, ep = model.get_loss(ep, sdf_weight=10., num_sample_points=100, FLAGS=F)
    assert set(ep["losses"]) >= {"accuracy", "sdf_loss", "sdf_loss_realvalue", "overall_loss"}
    feats = model.placeholder_features(2, 100)
    assert feats["point_img_feat"].shape == (2, 100, 1, 1472)


@pytest.mark.parametrize("flag", ["binary", "threedcnn", "img_feat_onestream", "multi_view", "alpha"])
def test_out_of_scope_branches_are_refused_loudly(flag):
    from disn_b200 import model_normalization as model
    F = _flags(**{flag: True})
    pls = model.placeholder_inputs(1, 1, (137, 137), num_sample_pc=8, FLAGS=_flags())
    with pytest.raises(NotImplementedError, match=flag):
        model.get_model(pls, 1, None, FLAGS=F)


def test_driver_constants_match_reference_arithmetic(golden, tmp_path):
    from disn_b200 import create_sdf as cs
    for sdf_res, R, total, split, nsp in golden["chunking"]["table"]:
        cs.configure(_flags(sdf_res=int(sdf_res), log_dir=str(tmp_path / ("log%d" % sdf_res))))
        assert (cs.RESOLUTION, cs.TOTAL_POINTS, cs.SPLIT_SIZE, cs.NUM_SAMPLE_POINTS) == (R, total, split, nsp)
        assert cs.RESULT_OBJ_PATH.endswith(os.path.join("test_objs", "%d_0.0" % R))
    from oracle import disn_oracle as orc
    cs.configure(_flags(sdf_res=6, log_dir=str(tmp_path / "g")))
    np.testing.assert_array_equal(cs.build_grid_points([-1, -1, -1, 1, 1, 1])[0],
                                  orc.grid_points([-1, -1, -1, 1, 1, 1], 7))


def test_dist_roundtrip_and_obj_writer(golden, tmp_path):
    from disn_b200 import create_sdf as cs
    g = golden["dist_roundtrip"]
    res = int(g["res"])
    fn = str(tmp_path / "t.dist")
    cs.to_binary(res, list(g["bbox"]), g["values"].astype(np.float64), fn)
    assert np.array_equal(np.fromfile(fn, dtype=np.uint8), g["file_bytes"])     # == reference reader's input
    r2, bbox, vals = cs.read_dist(fn)
    assert r2 == res and np.array_equal(vals.reshape(-1), g["values"]) and np.allclose(bbox, g["bbox"])
    # OBJ conventions of demo/result.obj: '# Number of vertices', 'v %g %g %g', 1-based faces
    v = np.array([[0.46875, -0.179688, -0.382966], [1, 2, 3], [0.5, 0.25, 1e-7]], np.float32)
    f = np.array([[0, 1, 2]], np.int32)
    on = str(tmp_path / "m.obj")
    cs.write_obj(on, v, f)
    lines = open(on).read().splitlines()
    assert lines[1] == "# Number of vertices: 3" and lines[2] == "# Number of faces: 1"
    assert lines[3] == "v 0.46875 -0.179688 -0.382966" and lines[-1] == "f 1 2 3"
    with pytest.raises(ValueError):
        open(fn, "ab").write(b"xx")
        cs.read_dist(fn)


def test_slab_partition_properties():
    from disn_b200 import sharding
    for R in (9, 65, 129, 257, 513):
        for world in (1, 2, 3, 4, 8):
            b = sharding.z_bounds(R, world)
            assert b[0] == 0 and b[-1] == R and all(b[i] <= b[i + 1] for i in range(world))
            sizes = [b[i + 1] - b[i] for i in range(world)]
            assert max(sizes) - min(sizes) <= 1 and max(sizes) == sharding.max_planes(R, world)
    assert sharding.z_bounds(257, 8) == [0, 32, 64, 96, 128, 160, 192, 224, 257]


def _gloo_worker(rank, world, R, port, outdir):
    import torch
    import torch.distributed as dist
    from disn_b200 import sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    z0, z1 = sharding.slab(R, world, rank)
    mp = sharding.max_planes(R, world)
    zz, yy, xx = torch.meshgrid(torch.arange(z0, z1), torch.arange(R), torch.arange(R), indexing="ij")
    slab = torch.zeros((mp, R, R))
    slab[:z1 - z0] = (zz * R * R + yy * R + xx).float()          # stand-in for the rank's SDF slab
    full = torch.empty((world * mp, R, R))
    dist.all_gather_into_tensor(full, slab)
    out = sharding.unpack_gathered(full, R, world, torch.empty((R, R, R)))
    # the bench's device path: gather (not all-gather) of the padded slabs to rank 0
    glist = [torch.empty_like(slab) for _ in range(world)] if rank == 0 else None
    dist.gather(slab, gather_list=glist, dst=0)
    # the bench's host path: every rank writes its slab into ONE shared host grid (file-backed shared memory)
    shm = os.path.join(outdir, "shared_grid.bin")
    if rank == 0:
        with open(shm, "wb") as f:
            f.truncate(R ** 3 * 4)
    dist.barrier()
    host = torch.from_file(shm, shared=True, size=R ** 3, dtype=torch.float32).view(R, R, R)
    host[z0:z1] = slab[:z1 - z0]
    dist.barrier()
    t = torch.tensor([float(rank + 1)])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)                      # the bench's max-over-ranks timing reduction
    if rank == 0:
        np.save(os.path.join(outdir, "gathered.npy"), sharding.unpack_gather_list(glist, R, world, torch.empty((R, R, R))).numpy())
        np.save(os.path.join(outdir, "shared.npy"), host.numpy().copy())
        np.save(os.path.join(outdir, "full.npy"), out.numpy())
        np.save(os.path.join(outdir, "tmax.npy"), t.numpy())
    dist.destroy_process_group()


@pytest.mark.parametrize("R", [9, 17])
def test_two_rank_slab_gather_gloo(R, tmp_path):
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() % 2000) + R
    mp.spawn(_gloo_worker, args=(2, R, port, str(tmp_path)), nprocs=2, join=True)
    full = np.load(tmp_path / "full.npy")
    np.testing.assert_array_equal(full.reshape(-1), np.arange(R ** 3, dtype=np.float32))
    np.testing.assert_array_equal(np.load(tmp_path / "gathered.npy"), full)
    np.testing.assert_array_equal(np.load(tmp_path / "shared.npy"), full)
    assert np.load(tmp_path / "tmax.npy")[0] == 2.0


def test_tf_checkpoint_bundle_round_trip(tmp_path):
    """tensor-bundle writer -> reader round trip with the path's variable names/shapes (format restated from
    TensorFlow's tensor_bundle; unpinned against a real checkpoint, see disn_b200/tf_checkpoint.py)."""
    from disn_b200 import synth
    from disn_b200 import tf_checkpoint as ck
    rng = np.random.default_rng(0)
    shapes = {k: v for k, v in synth.weight_shapes().items() if "fc6" not in k and "fc7" not in k}
    tensors = {k: rng.standard_normal(v).astype(np.float32) for k, v in list(shapes.items())[:40]}
    tensors["global_step"] = np.array(12345, dtype=np.int64)
    prefix = str(tmp_path / "ckpt" / "model.ckpt")
    ck.save_checkpoint(prefix, tensors)
    idx = ck.read_index(prefix + ".index")
    assert set(idx) == set(tensors)
    assert idx["vgg_16/conv1/conv1_1/weights"]["shape"] == (3, 3, 3, 64)
    got = ck.load_checkpoint(prefix, prefixes=("vgg_16/", "sdfprediction"))
    assert "global_step" not in got and len(got) == len(tensors) - 1
    for k, v in got.items():
        np.testing.assert_array_equal(v, tensors[k])
    with pytest.raises(ValueError, match="bad table magic"):
        open(prefix + ".bad.index", "wb").write(b"x" * 100)
        ck.read_index(prefix + ".bad.index")


def test_demo_image_loader_and_gt_camera(tmp_path):
    """demo/demo.py:261-279: PNG -> [1,137,137,3] float32 in [0,1] (alpha dropped), the hard-coded GT trans_mat and
    sdf_params = [-1,-1,-1,1,1,1]."""
    import cv2
    from disn_b200 import create_sdf as drv
    from disn_b200 import demo, synth
    drv.configure(demo.default_flags(log_dir=str(tmp_path)))
    img = (np.random.default_rng(0).random((137, 137, 4)) * 255).astype(np.uint8)
    path = str(tmp_path / "render.png")
    cv2.imwrite(path, img)
    bd = demo.read_img_get_transmat(path)
    np.testing.assert_array_equal(bd["img"][0], img[:, :, :3].astype(np.float32) / 255.)
    np.testing.assert_array_equal(bd["trans_mat"], synth.DEMO_TRANS_MAT)
    np.testing.assert_array_equal(bd["sdf_params"], [[-1, -1, -1, 1, 1, 1]])
    with pytest.raises(FileNotFoundError):
        demo.read_img_get_transmat(str(tmp_path / "missing.png"))
    with pytest.raises(RuntimeError):           # --cam_est without the camera checkpoint's variables
        demo.read_img_get_transmat(path, cam_est=True)


def test_tf_checkpoint_reader_against_independently_assembled_bundle(tmp_path):
    """The reader is pinned by a bundle assembled byte by byte from the documented table layout by tests/tf_bundle_golden.py
    (no code shared with the module's writer): prefix-compressed keys, 16-entry restarts, several blocks, shortened index
    keys, two data shards, optimizer slots + global_step; plus crc32c known answers and the loud failure modes."""
    import struct
    from disn_b200 import synth, tf_checkpoint as ck
    from tests import tf_bundle_golden as gb
    # crc32c known-answer vectors (RFC 3720 B.4) for both implementations
    kat = [(b"123456789", 0xE3069283), (bytes(32), 0x8A9136AA), (b"\xff" * 32, 0x62A8AB43), (bytes(range(32)), 0x46DD794E),
           (bytes(range(31, -1, -1)), 0x113FDB5C)]
    for data, want in kat:
        assert gb.crc32c_bitwise(data) == want and ck.crc32c(data) == want
    assert ck._masked_crc32c(b"123456789") == gb.mask(0xE3069283)
    rng = np.random.default_rng(0)
    shapes = {k: v for k, v in synth.weight_shapes().items() if "fc6" not in k and "fc7" not in k}   # keep it small
    tensors = {}
    for name, shp in shapes.items():
        small = tuple(min(d, 6) for d in shp)                 # many entries, few bytes
        tensors[name] = rng.standard_normal(small).astype(np.float32)
        if name.endswith("weights"):
            tensors[name + "/Adam"] = np.zeros(small, np.float32)
            tensors[name + "/Adam_1"] = np.zeros(small, np.float32)
    tensors["global_step"] = np.array(123456, np.int64)
    tensors["beta1_power"] = np.array(0.5, np.float32)
    prefix = str(tmp_path / "model.ckpt")
    shard_of = lambda n: 1 if n.startswith("sdfprediction_imgfeat") else 0
    idx = gb.write_bundle(prefix, tensors, num_shards=2, shard_of=shard_of, block_size=512)
    entries, header = ck.read_index(prefix + ".index", with_header=True)
    assert header == dict(num_shards=2, endianness=0, version=1)
    assert set(entries) == set(tensors) and len(idx) > 6 * 512             # several data blocks, multi-entry index block
    assert entries["sdfprediction_imgfeat/fold2/conv1/weights"]["shard_id"] == 1
    got = ck.load_checkpoint(prefix, prefixes=("vgg_16/", "sdfprediction"), verify_data=True)
    want = {k: v for k, v in tensors.items() if ck.is_model_variable(k) and k.startswith(("vgg_16/", "sdfprediction"))}
    assert set(got) == set(want) and not any(k.endswith(("/Adam", "/Adam_1")) for k in got)
    for k in want:
        np.testing.assert_array_equal(got[k], want[k])
    everything = ck.load_checkpoint(prefix, model_variables_only=False)
    assert everything["global_step"] == 123456 and "vgg_16/conv1/conv1_1/weights/Adam_1" in everything
    # the module's own writer must produce something this reader AND the independent expectations agree on
    ck.save_checkpoint(str(tmp_path / "own.ckpt"), {k: tensors[k] for k in list(want)[:20]})
    own = ck.read_index(str(tmp_path / "own.ckpt.index"))
    for k, e in own.items():
        assert e["crc32c"] == gb.mask(gb.crc32c_bitwise(tensors[k].tobytes()))
    # failure modes are loud: snappy-flagged blocks, a flipped byte in a data block, a truncated shard, a corrupted tensor
    gb.write_bundle(str(tmp_path / "snappy.ckpt"), want, compression_type=1)
    with pytest.raises(NotImplementedError, match="snappy"):
        ck.read_index(str(tmp_path / "snappy.ckpt.index"))
    bad = bytearray(idx)
    bad[100] ^= 0x40
    open(str(tmp_path / "bad.ckpt.index"), "wb").write(bytes(bad))
    with pytest.raises(ValueError, match="crc32c"):
        ck.read_index(str(tmp_path / "bad.ckpt.index"))
    d0 = prefix + ".data-00000-of-00002"
    raw = open(d0, "rb").read()
    open(d0, "wb").write(raw[:-16])
    with pytest.raises(ValueError, match="truncated"):
        ck.load_checkpoint(prefix, model_variables_only=False)
    flipped = bytearray(raw)
    flipped[5] ^= 1
    open(d0, "wb").write(bytes(flipped))
    with pytest.raises(ValueError, match="crc32c"):
        ck.load_checkpoint(prefix, verify_data=True, model_variables_only=False)


def test_bench_contract_helpers(tmp_path):
    """bench.py: both arms print the same config.workload for every BASELINE config, the clock sampler degrades to a
    one-shot sample / 'unavailable' without nvidia-smi, the z-slab bookkeeping of the host path covers the grid, and
    --dump-outputs writes a small grid whole and a large one as the same seeded float sample every time."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(os.path.dirname(os.path.dirname(__file__)), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.workload_string(1) == "single 137x137 image, --sdf_res 256 (257^3 = 16974593 points), twostream, encoder included per step"
    assert bench.workload_string(0).startswith("single 137x137 image, --sdf_res 64 (65^3 = 274625 points)")
    assert bench.workload_string(2).startswith("batch of 8 137x137 images, --sdf_res 128 (8 x 129^3 = 17173512 points)")
    assert bench.workload_string(4).startswith("single 137x137 image, --sdf_res 512 (513^3 = 135005697 points)")
    assert abs(bench.F_ALG - 2 * 2 * (3 * 64 + 64 * 256 + 256 * 512 + 512 * 512 + 512 * 256 + 256)) < 1e-9
    s = bench.ClockSampler(0, period_ms=0)
    s.start()
    out = s.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    from disn_b200 import sharding
    for world in (1, 2, 4, 8):
        b = sharding.z_bounds(257, world)
        assert sum(b[i + 1] - b[i] for i in range(world)) == 257
    small = np.random.default_rng(1).standard_normal((1, 9, 9, 9)).astype(np.float32)
    bench.dump_outputs(str(tmp_path / "small"), small)
    assert os.listdir(tmp_path / "small") == ["sdf.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "small" / "sdf.npy"), small)
    large = np.arange(bench.DUMP_FULL_BYTES // 4 + 1, dtype=np.float32)
    for d in ("large", "again"):
        bench.dump_outputs(str(tmp_path / d), large, mesh_counts=(10, 20))
    files = sorted(os.listdir(tmp_path / "large"))
    assert files == ["mesh_counts.npy", "sdf_sample.npy", "sdf_sample_index.npy"]
    assert sum(os.path.getsize(tmp_path / "large" / f) for f in files) <= 64 << 20
    got = {f: np.load(tmp_path / "large" / f) for f in files}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert got["sdf_sample.npy"].shape == (bench.DUMP_SAMPLE,)
    np.testing.assert_array_equal(got["sdf_sample.npy"], large[got["sdf_sample_index.npy"].astype(np.int64)])
    np.testing.assert_array_equal(got["mesh_counts.npy"], [10, 20])
    for f in files:
        np.testing.assert_array_equal(np.load(tmp_path / "again" / f), got[f])
