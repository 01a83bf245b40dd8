"""Host-side logic that must work without a GPU."""
import argparse

import numpy as np
import pytest
import torch

from read_b200 import synth, dist as rdist, ops
from read_b200.unet import UNet, layer_table
from read_b200.texture import PointTexture
from read_b200.compose import NetAndTexture
from read_b200.pipeline import TexturePipeline


def test_layer_table_counts():
    t = layer_table()
    assert len(t) == 101                                  # 99 used by forward + 2 unused ConvsOut (unet.py:181-186)
    net = UNet()
    assert len(net.state_dict()) == 909                   # SURVEY.md §5
    assert sum(p.numel() for p in net.parameters()) == 30193988


def test_synth_state_dict_loads_strict_and_is_deterministic(synth_sd):
    UNet().load_state_dict(synth_sd, strict=True)
    again = synth.synth_state_dict(synth.SEED)
    assert all(torch.equal(synth_sd[k], again[k]) for k in synth_sd)


def test_proj_matrix_restatement():
    K = synth.intrinsics(640, 480)
    P = synth.get_proj_matrix(K, (640, 480), 0.1, 1000.0)
    assert P.shape == (4, 4)
    assert P[3, 2] == -1.0 and P[3, 3] == 0.0             # returned transposed: w_clip = -z_eye
    assert abs(P[0, 0] - 2 * 0.8) < 1e-12 and abs(P[1, 1] - 2 * 0.8 * 640 / 480) < 1e-12
    assert abs(P[2, 2] - (1000.1 / -999.9)) < 1e-12


def test_street_scene_shape_and_determinism():
    a = synth.street_scene(10000)
    b = synth.street_scene(10000)
    assert a.shape == (10000, 3) and a.dtype == np.float32 and np.array_equal(a, b)
    assert a[:, 2].min() >= -250 - 5 and a[:, 2].max() <= 5


def test_inference_on_cpu_raises_no_silent_fallback(synth_sd):
    net = UNet().eval()
    xs = [torch.zeros(1, 8, 32 >> l, 32 >> l) for l in range(4)]
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        net(*xs)
    tex = PointTexture(8, 10, init_method='rand')
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        tex(torch.zeros(1, 1, 4, 4))


def test_net_and_texture_texture_management():
    net = UNet()
    texs = {0: PointTexture(8, 10), 3: PointTexture(8, 20)}
    m = NetAndTexture(net, texs, supersampling=1)
    assert m.ss == 1 and m.temporal_average is False and m.last_input is None
    m.load_textures([3])
    assert '3' in m._modules and any(n == '3.texture_' for n, _ in m.named_parameters())
    assert m.reg_loss() == 0
    m.unload_textures()
    assert '3' not in m._modules
    m.load_textures(torch.tensor([0, 3]))
    assert m._loaded_textures == [0, 3]


def test_pipeline_exports_reference_flags_and_creates_inference_model():
    class P(argparse.ArgumentParser):
        add = argparse.ArgumentParser.add_argument
    parser = P()
    pipe = TexturePipeline()
    pipe.export_args(parser)
    a = parser.parse_args([])
    assert a.descriptor_size == 8 and a.texture_lr == 0.1 and a.texture_activation == 'none' and a.n_points == 0
    a.inference, a.n_points, a.use_mesh, a.num_mipmap = True, 123, False, 5
    pipe.create(a)
    assert isinstance(pipe.model, NetAndTexture) and pipe.get_net() is pipe.net
    assert pipe.textures[0].texture_.shape == (1, 8, 123)


def test_level_sizes_helper():
    assert ops.level_sizes(1920, 1080, 5) == [(1920, 1080), (960, 540), (480, 270), (240, 135), (120, 67)]


def test_shard_ranges_cover_and_align():
    for n in (0, 1, 1023, 1024, 10_000_000, 123_457):
        for ws in (1, 2, 4, 8):
            spans = [rdist.shard_range(n, r, ws) for r in range(ws)]
            assert sum(c for _, c in spans) == n
            pos = 0
            for s, c in spans:
                assert s == pos or c == 0
                assert s % 1024 == 0 or c == 0
                pos = s + c


def test_reduce_span_only_covers_direct_levels():
    sizes = ops.level_sizes(64, 32, 4)
    offs, o = [], 0
    for (w, h) in sizes:
        offs.append(o)
        o += 2 * w * h
    assert rdist.reduce_span(offs, sizes, 2, [0]) == (0, 2 * 64 * 32)
    assert rdist.reduce_span(offs, sizes, 2, [0, 3]) == (0, o)


def test_sorted_points_store_is_a_spatially_coherent_permutation():
    """ops.SortedPoints (scene-load preprocessing, plain torch): a permutation of the cloud in Morton order of 3-D grid cells
    with the ORIGINAL ids carried as bit patterns; contiguous ranges (the multi-GPU shards) are compact spatial tiles."""
    import numpy as np
    import torch
    from read_b200 import ops, synth
    n = 50_000
    xyz = torch.from_numpy(synth.street_scene(n, depth=60.0, seed=9))
    st = ops.SortedPoints(xyz, cell=0.5)
    assert st.n == n and tuple(st.pts4.shape) == (n, 4) and st.pts4.dtype == torch.float32
    assert torch.equal(torch.sort(st.perm).values, torch.arange(n))                       # a permutation
    assert torch.equal(st.pts4[:, :3], xyz[st.perm])                                      # coordinates untouched
    ids = st.pts4[:, 3].contiguous().view(torch.int32).to(torch.int64)
    assert torch.equal(ids, st.perm)                                                      # original ids, bit-exact
    # ties inside a cell keep the original order (stable sort): ids ascend within equal cells
    q = torch.floor((xyz - xyz.min(0).values) / 0.5).to(torch.int64)[st.perm]
    same = (q[1:] == q[:-1]).all(1)
    assert bool((ids[1:][same] > ids[:-1][same]).all())
    # spatial coherence: consecutive rows are (much) closer than consecutive rows of the generator order
    d_sorted = (st.pts4[1:, :3] - st.pts4[:-1, :3]).norm(dim=1).median()
    d_orig = (xyz[1:] - xyz[:-1]).norm(dim=1).median()
    assert float(d_sorted) < 0.25 * float(d_orig)
    # a shard = contiguous range of the Morton order = a spatial tile: a view (no copy), and much more compact than a random
    # subset of the same size (a Morton range may straddle one coarse cell boundary, so compare spreads, not boxes)
    sh = st.shard(1024 * 8, 1024 * 4)
    assert sh.n == 4096 and sh.pts4.data_ptr() == st.pts4[1024 * 8:].data_ptr()
    assert float(sh.pts4[:, 2].std()) < 0.5 * float(xyz[:, 2].std())
    with pytest.raises(RuntimeError, match="float"):
        ops.SortedPoints(xyz.double())
    assert ops.SortedPoints(torch.empty((0, 3))).n == 0


def test_bench_dump_outputs_writes_float_arrays_within_the_size_limit(tmp_path):
    import bench
    rgb = np.arange(6, dtype=np.float16).reshape(1, 2, 3)
    bench.dump_outputs(str(tmp_path / "d"), {"rgb": rgb, "loss": np.float64(0.25)})
    got = np.load(tmp_path / "d" / "rgb.npy")
    assert got.dtype == np.float32 and np.array_equal(got, rgb.astype(np.float32))
    assert np.load(tmp_path / "d" / "loss.npy").dtype == np.float64
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "e"), {"rgb": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "e").exists()
