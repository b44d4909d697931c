"""CPU-side tests: C-ABI surface, host logic, error behaviour, multi-process sharding (gloo)."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest
import torch

from tests.conftest import ROOT, load_golden


def test_library_loads_and_exports_every_declared_symbol():
    from pointmvsnet_b200 import _lib
    header = open(os.path.join(ROOT, "include", "pmvs_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(pmvs_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(_lib.lib, name), "libpmvs_b200.so does not export %s" % name
    assert set(_lib.EXPORTED) == set(declared)
    assert _lib.lib.pmvs_version() >= 100


def test_argument_errors_are_reported_without_touching_the_gpu():
    from pointmvsnet_b200 import _lib
    lib = _lib.lib
    dummy = C.c_void_p(256)
    # unsupported knn / kernel size -> PMVS_ERR_ARG + message (checked before any launch)
    assert lib.pmvs_knn3d(dummy, dummy, None, 1, 5, 8, 8, 5, 7, None) == 1
    assert b"unsupported knn" in lib.pmvs_last_error()
    assert lib.pmvs_knn3d(dummy, dummy, None, 1, 5, 8, 8, 4, 16, None) == 1
    assert lib.pmvs_knn3d(dummy, dummy, dummy, 1, 5, 8, 8, 5, 16, None) == 1  # both outputs given
    assert lib.pmvs_knn3d(dummy, dummy, None, 1, 1, 2, 2, 3, 32, None) == 1  # knn > window
    with pytest.raises(RuntimeError):
        _lib.check(lib.pmvs_gather_knn_forward(None, None, None, 1, 1, 1, 1, None))
    assert lib.pmvs_gather_knn_forward(None, None, None, 1, 2, 0, 4, None) == 0  # empty input is fine
    s = _lib.FlowShape()
    s.B, s.V = 1, 99
    assert lib.pmvs_point_flow_workspace_bytes(C.byref(s)) == 0
    assert b"V" in lib.pmvs_last_error()


def test_workspace_plan_sizes():
    from pointmvsnet_b200 import _lib
    from pointmvsnet_b200.point_flow import PointFlow
    s = PointFlow.make_shape(1, 4, [(256, 320), (128, 160), (64, 80)], (128, 160), (512, 640), 0.5, True)
    assert (s.flow_h, s.flow_w, s.ratio) == (256, 320, 4)
    need = _lib.lib.pmvs_point_flow_workspace_bytes(C.byref(s))
    rows = 16 * 25600
    assert need >= rows * (136 + 3 + 16 + 128 + 224 + 64 + 64 + 16) * 4
    assert need < rows * 800 * 4  # includes the [B,V,h,w,112] warp source map (model.py:184)
    off = (C.c_size_t * 10)()
    assert _lib.lib.pmvs_point_flow_debug_offsets(C.byref(s), C.byref(off)) == 0
    assert all(o % 256 == 0 for o in list(off)[:9]) and off[9] in (0, 1)
    # divisibility required by the sub-grid view (model.py:240-243)
    bad = PointFlow.make_shape(1, 4, [(256, 320), (128, 160), (64, 80)], (64, 80), (514, 640), 0.5, True)
    assert _lib.lib.pmvs_point_flow_workspace_bytes(C.byref(bad)) == 0


def test_ratio_rule_follows_reference():
    from pointmvsnet_b200.point_flow import _ratio_for
    assert [_ratio_for(s, True) for s in (0.125, 0.25, 0.5, 1.0)] == [1, 2, 4, 8]
    assert _ratio_for(0.25, False) == 1  # train branch: one cloud (model.py:271)
    with pytest.raises(NotImplementedError):  # model.py:268
        _ratio_for(0.3, True)


def test_state_dict_names_match_reference_checkpoint(golden_weights):
    from pointmvsnet_b200.point_flow import PointFlow
    pf = PointFlow()
    own = pf.state_dict()
    assert set(own.keys()) == set(golden_weights.keys())
    for k, v in golden_weights.items():
        assert tuple(own[k].shape) == tuple(v.shape), k
    pf.load_reference_state_dict({"module." + k: v for k, v in golden_weights.items()})
    assert torch.equal(pf.flow_mlp[1].weight, golden_weights["flow_mlp.1.weight"])
    broken = dict(golden_weights)
    del broken["flow_mlp.0.1.conv.weight"]
    with pytest.raises(KeyError):
        PointFlow().load_reference_state_dict(broken)
    broken = dict(golden_weights)
    broken["flow_edge_conv.0.conv1.weight"] = torch.zeros(32, 128, 1)
    with pytest.raises(ValueError):
        PointFlow().load_reference_state_dict(broken)


def test_no_cpu_fallback():
    from pointmvsnet_b200.utils.feature_fetcher import FeatureFetcher
    from pointmvsnet_b200.utils.torch_utils import get_knn_3d
    from pointmvsnet_b200.networks import EdgeConv
    from pointmvsnet_b200.functions.gather_knn import gather_knn
    with pytest.raises(RuntimeError):
        get_knn_3d(torch.zeros(1, 3, 5, 4, 4), 5, 16)
    with pytest.raises(RuntimeError):
        FeatureFetcher()(torch.zeros(1, 1, 4, 8, 8), torch.zeros(1, 3, 2), torch.eye(3).view(1, 1, 3, 3), None)
    with pytest.raises(RuntimeError):
        with torch.no_grad():
            EdgeConv(32, 32)(torch.zeros(1, 32, 10), torch.zeros(1, 10, 16, dtype=torch.long))
    with pytest.raises(RuntimeError):
        gather_knn(torch.zeros(1, 2, 3), torch.zeros(1, 3, 2, dtype=torch.long))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pointmvsnet_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("oracle-style", ""), f


def test_install_as_pointmvsnet_aliases():
    import pointmvsnet_b200
    saved = {k: v for k, v in sys.modules.items() if k == "pointmvsnet" or k.startswith("pointmvsnet.")}
    try:
        pointmvsnet_b200.install_as_pointmvsnet()
        from pointmvsnet.utils.torch_utils import get_knn_3d as a  # noqa
        from pointmvsnet_b200.utils.torch_utils import get_knn_3d as b
        assert a is b
        from pointmvsnet.functions import dgcnn_ext  # noqa
        assert hasattr(dgcnn_ext, "gather_knn_forward") and hasattr(dgcnn_ext, "gather_knn_backward")
        # output side (test.py:19,76; dataset.py:114,122): the reference's module and function names
        import pointmvsnet.utils.io as ref_io  # noqa
        from pointmvsnet.utils.eval_file_logger import eval_file_logger  # noqa
        for fn in ("mkdir", "load_cam_dtu", "write_cam_dtu", "load_pfm", "write_pfm"):
            assert callable(getattr(ref_io, fn))
        assert eval_file_logger.__module__ == "pointmvsnet_b200.utils.eval_file_logger"
    finally:
        for k in [k for k in sys.modules if k == "pointmvsnet" or k.startswith("pointmvsnet.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_synthetic_generator_is_deterministic_and_dtu_shaped():
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    a = make_pointflow_inputs(64, 128, 3, 1, 48, seed=3)
    b = make_pointflow_inputs(64, 128, 3, 1, 48, seed=3)
    assert all(torch.equal(x, y) for x, y in zip(a["pyramids"], b["pyramids"]))
    assert [tuple(p.shape) for p in a["pyramids"]] == [(1, 3, 16, 32, 64), (1, 3, 32, 16, 32), (1, 3, 64, 8, 16)]
    cams = a["cam_params_list"]
    assert tuple(cams.shape) == (1, 3, 2, 4, 4)
    R = cams[0, :, 0, :3, :3]
    assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3).expand(3, 3, 3), atol=1e-5)
    assert abs(cams[0, 0, 1, 3, 1].item() - 2.5 * 4.24) < 1e-5  # config.py:28


def test_shard_views_partition():
    from pointmvsnet_b200.parallel import shard_views
    for n, w in ((49, 8), (7, 2), (3, 4), (8, 8)):
        parts = [shard_views(n, r, w) for r in range(w)]
        assert sum(parts, []) == list(range(n))
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from pointmvsnet_b200.parallel import shard_views, gather_depth_maps, gather_ragged_depth_maps, gather_view_pyramids
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
views = 5
mine = shard_views(views, rank, world)
local = torch.stack([torch.full((1, 4, 6), float(v)) for v in mine])  # "depth map" of view v is v everywhere
full = gather_ragged_depth_maps(local, views)
assert full.shape == (views, 1, 4, 6)
assert torch.equal(full[:, 0, 0, 0], torch.arange(views, dtype=torch.float32)), full[:, 0, 0, 0]
eq = gather_depth_maps(torch.full((1, 1, 4, 6), float(rank)))
assert [t[0, 0, 0, 0].item() for t in eq] == [float(r) for r in range(world)]
# C5 view-sharded input: every rank owns some views' pyramids, one all-gather per level gives everyone all V
V = 5
g = torch.Generator().manual_seed(3)
full_pyr = [torch.randn(1, V, c, 4, 6, generator=g) for c in (16, 32, 64)]
own = shard_views(V, rank, world)
got = gather_view_pyramids([lv[:, own] for lv in full_pyr], V, rank, world)
assert all(torch.equal(a, b) for a, b in zip(got, full_pyr))
# C5 latency split: SubCloudShardedPass drives a point-flow callable per iteration with this rank's range of
# sub-clouds and re-assembles the map with one all-reduce.  A CPU stand-in for the fused module (writes a value that
# encodes iteration, sub-cloud and the previous depth into exactly the pixels of the requested sub-clouds) checks the
# control flow: every rank ends with the map a single process computes.
from pointmvsnet_b200.parallel import SubCloudShardedPass
import torch.nn.functional as F
class FakeFlow(object):
    update_running_stats = True
    def __call__(self, depth, interval, scale, it, out=None, sub_range=None, img_hw=None, **kw):
        r = int(scale * 8)
        h, w = int(img_hw[0] * scale), int(img_hw[1] * scale)
        prev = F.interpolate(depth, (h, w), mode="nearest")
        first, count = sub_range if sub_range is not None else (0, r * r)
        ys = torch.arange(h).view(h, 1).expand(h, w)
        xs = torch.arange(w).view(1, w).expand(h, w)
        sid = (ys %% r) * r + (xs %% r)
        mine = (sid >= first) & (sid < first + count)
        val = prev[:, 0] * 2.0 + 1000.0 * (it + 1) + sid.float()
        out[0][:, 0][:, mine] = val[:, mine]
        return out
img_hw = (32, 48)
coarse = torch.arange(4 * 6, dtype=torch.float32).view(1, 1, 4, 6)
single = SubCloudShardedPass(FakeFlow(), 0, 1).run(None, coarse, None, None, None, None, img_hw)
ff = FakeFlow()
sharded = SubCloudShardedPass(ff, rank, world).run(None, coarse, None, None, None, None, img_hw)
assert ff.update_running_stats is False
assert sharded.shape == (1, 1, 16, 24) and torch.equal(sharded, single), (sharded - single).abs().max()
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_depth_map_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % ROOT)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29531")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=120)
        assert p.returncode == 0 and "OK" in out, out


def test_sub_cloud_partition_covers_every_unit_once():
    """C5 partition (SURVEY 8e): 1 / 4 / 16 sub-clouds over 1, 2, 4, 8 ranks - every sub-cloud exactly once,
    contiguous blocks, iteration 1 replicated; the 8-rank critical path is 1 + 1 + 2 units."""
    from pointmvsnet_b200.parallel import shard_sub_clouds
    for world in (1, 2, 4, 8):
        for S in (4, 16):
            owned = []
            for r in range(world):
                first, count = shard_sub_clouds(S, r, world)
                owned += list(range(first, first + count))
            assert sorted(owned) == list(range(S))
        assert all(shard_sub_clouds(1, r, world) == (0, 1) for r in range(world))
    assert max(shard_sub_clouds(16, r, 8)[1] for r in range(8)) == 2
    assert max(shard_sub_clouds(4, r, 8)[1] for r in range(8)) == 1


def test_bench_algorithmic_bytes_match_survey():
    sys.path.insert(0, ROOT)
    import bench
    alg = bench.algorithmic_bytes_per_pass(512, 640, 4)
    # SURVEY.md section 8d: C2 fetch traffic 51.0 / 93.7 / 264.8 MB per iteration (sum 409.5 MB)
    assert abs(alg["fused_fetch"][0] / 1e6 - 409.5) < 1.0
    assert alg["fused_fetch"][1] == 3
    assert alg["knn3d"][0] == 537600 * 76
    # the stage numerators of `roofline_stage` are SURVEY 8(d)'s: 409.5 MB fetch, 140 B/pt kNN (75 MB), 3 108 B/pt
    # EdgeConv + MLP (1.67 GB) for one C2 pass
    surv = bench.survey_8d_bytes_per_pass(512, 640, 4)
    assert abs(surv["fetch"] / 1e6 - 409.5) < 1.0
    assert surv["knn"] == 537600 * 140 and surv["edgeconv_mlp"] == 537600 * 3108


def test_bench_per_iteration_grouping():
    sys.path.insert(0, ROOT)
    import bench
    one_iter = [("cam_setup", 0.01), ("warp_source", 0.1), ("fused_fetch", 0.2), ("knn3d", 0.3)]
    one_pass = [("transpose", 1.0)] * 3 + one_iter + [(n, 2 * m) for n, m in one_iter] + [(n, 4 * m) for n, m in one_iter]
    ms = bench.per_iteration_kernel_ms(one_pass * 5, 3)
    assert ms == pytest.approx([0.61, 1.22, 2.44])
    assert bench.per_iteration_kernel_ms(one_pass[:-4], 3) is None   # truncated pass
    assert bench.per_iteration_kernel_ms([("knn3d", 1.0)], 3) is None


def test_unchanged_reference_model_imports_our_operators(tmp_path):
    """Drop-in check against what the reference's UNCHANGED pointmvsnet/model.py resolved (tests/golden/
    dropin_model.json, written by tests/golden/make_golden_dropin.py from a checkout and its pretrained checkpoint).
    install_as_pointmvsnet(reference_root) - here over empty stand-ins of the checkout's modules - and the stub mode
    without a checkout both hand out our object for every name model.py took from this package (model.py:8-12);
    the submodules PointMVSNet built from our classes have the checkpoint's layout, and PointFlow builds them under
    the same names or runs on a model's own modules."""
    import importlib
    import json
    import pointmvsnet_b200
    from pointmvsnet_b200.point_flow import PointFlow
    with open(os.path.join(ROOT, "tests", "golden", "dropin_model.json")) as f:
        g = json.load(f)

    def resolve(path):
        mod, qual = path.split(":")
        return getattr(importlib.import_module(mod), qual)

    for name, kind in g["reference_modules"].items():
        p = tmp_path.joinpath(*name.split("."))
        if kind == "package":
            p.mkdir(parents=True, exist_ok=True)
            (p / "__init__.py").write_text("")
        else:
            p.parent.mkdir(parents=True, exist_ok=True)
            p.with_suffix(".py").write_text("")
    assert g["imports"]

    def drop_aliases():
        for k in [k for k in sys.modules if k == "pointmvsnet" or k.startswith("pointmvsnet.")]:
            del sys.modules[k]

    saved = {k: v for k, v in sys.modules.items() if k == "pointmvsnet" or k.startswith("pointmvsnet.")}
    saved_path = list(sys.path)
    try:
        for root in (str(tmp_path), None):
            drop_aliases()
            pointmvsnet_b200.install_as_pointmvsnet(root)
            for name, rec in g["imports"].items():
                obj = resolve(rec["object"])
                for mod in rec["from"]:
                    assert getattr(importlib.import_module(mod), name, None) is obj, (root, mod, name)
    finally:
        drop_aliases()
        sys.modules.update(saved)
        sys.path[:] = saved_path
    pf = PointFlow()
    own = dict(pf.named_modules())
    assert g["submodules"]
    for path, rec in g["submodules"].items():
        cls = resolve(rec["class"])
        mod = own[path] if path in own else cls()
        assert type(mod) is cls, path
        assert {k: list(v.shape) for k, v in mod.state_dict().items()} == rec["state"], path
    shared = PointFlow(flow_edge_conv=pf.flow_edge_conv, flow_mlp=pf.flow_mlp)
    assert shared.flow_mlp[1].weight is pf.flow_mlp[1].weight


def test_image_conv_producer_names_layout_and_probability_map():
    """Row f1 on the CPU: ImageConv keeps the reference's parameter names (networks.py:84-111), its channels-last
    outputs stack into [B,V,h,w,C] memory, and get_propability_map (functions.py:141-175) sums the two bracketing
    planes."""
    import torch
    from pointmvsnet_b200.networks import ImageConv, stack_views_channels_last
    from pointmvsnet_b200.functions.functions import get_propability_map
    m = ImageConv(8)
    keys = list(m.state_dict().keys())
    assert len(keys) == 61 and keys[0] == "conv0.0.conv.weight" and keys[-1] == "conv3.2.weight"
    assert "conv1.0.bn.running_mean" in keys and m.out_channels == 64
    assert m.conv1[0].conv.kernel_size == (5, 5) and m.conv1[0].conv.stride == (2, 2)
    x = torch.randn(2, 3, 32, 40)
    per_view = [m(x) for _ in range(3)]
    stacked = stack_views_channels_last(per_view)
    for k, c, s in (("conv1", 16, 2), ("conv2", 32, 4), ("conv3", 64, 8)):
        t = stacked[k]
        assert tuple(t.shape) == (2, 3, c, 32 // s, 40 // s) and t.permute(0, 1, 3, 4, 2).is_contiguous()
        assert torch.equal(t[:, 1], per_view[1][k])
    cv = torch.zeros(1, 4, 1, 3)
    cv[0, :, 0, :] = torch.tensor([[.1, .2, .3], [.2, .3, .4], [.3, .4, .2], [.4, .1, .1]])
    depth = torch.tensor([10.5, 12.0, 99.0]).view(1, 1, 1, 3)  # between planes 0/1, exactly plane 2, beyond the last
    pm = get_propability_map(cv, depth, torch.tensor([10.0]), torch.tensor([1.0]))
    assert torch.allclose(pm.view(-1), torch.tensor([.1 + .2, .4 + .4, .1 + .1]))


def test_deterministic_gather_backward_workspace_size_is_host_only():
    """pmvs_gather_knn_backward_det_workspace_bytes is plain host arithmetic (callable without a GPU): two int32 arrays
    of B*N counters, B*(N+1) offsets and B*N*K list entries, each 256-byte aligned."""
    from pointmvsnet_b200 import _lib
    f = _lib.lib.pmvs_gather_knn_backward_det_workspace_bytes
    assert f(0, 0, 0) >= 0 and f(-1, 4, 4) == 0
    B, N, K = 2, 1200, 16
    need = 4 * (2 * B * N + B * (N + 1) + B * N * K)
    assert need <= f(B, N, K) <= need + 5 * 256
    assert f(1, 102400, 16) > f(1, 25600, 16) > 0
