"""GPU parity tests: the CUDA path (through the C ABI / Python mirror) against the CPU oracle
and the committed golden vectors.  Tolerances (fp32, stated per stage; measured errors on
B200 are ~10x smaller, see profiles/parity_r01.md):

  gather_knn fwd/bwd ............ bit exact
  FeatureFetcher vs oracle ...... atol 1e-5 (same op sequence; measured 0)
  kNN indices ................... bit exact on EVERY point (canonical tie order on both sides)
  variance features ............. atol 3e-5 + rtol 1e-5   (values up to ~6; cancellation)
  normalised xyz ................ atol 1e-6
  EdgeConv / EdgeConvNoC ........ atol 2e-5 + rtol 1e-4   (fp32 FMA order)
  depth after one iteration ..... atol 5e-4 mm (< 5e-5 * interval; depths ~650 mm, ulp 6e-5)
  flow probabilities ............ atol 5e-5
"""
import numpy as np
import pytest
import torch

from oracle import pointflow_oracle as O
from tests.conftest import load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pf(weights):
    from pointmvsnet_b200.point_flow import PointFlow
    pf = PointFlow().to(DEV)
    pf.load_reference_state_dict(weights)
    pf.train()
    return pf


def sub_to_ref(t, S, B, M, hs, ws, r):
    Cc = t.shape[-1]
    x = t.view(r, r, B, M, hs, ws, Cc).permute(2, 6, 3, 4, 0, 5, 1)
    return x.reshape(B, Cc, M, hs * r, ws * r)


def test_native_library_is_loaded():
    from pointmvsnet_b200 import _lib
    assert _lib.lib.pmvs_version() >= 100
    maps = open("/proc/self/maps").read()
    assert "libpmvs_b200.so" in maps


def test_gather_knn_golden_forward_backward():
    from pointmvsnet_b200.functions.gather_knn import gather_knn
    g = load_golden("gather_knn.npz")
    f = g["feature"].to(DEV).requires_grad_(True)
    out = gather_knn(f, g["index"].to(DEV))
    assert torch.equal(out.cpu(), g["out"])
    out.backward(g["grad_out"].to(DEV))
    assert torch.allclose(f.grad.cpu(), g["grad_in"], atol=1e-6)
    # reference's own inline test (gather_knn.py:27-56): equals torch.gather, grads of ones
    torch.manual_seed(1)
    feat = torch.rand(2, 4, 5, device=DEV)
    idx = torch.randint(0, 5, [2, 5, 3], device=DEV)
    a = feat.clone().requires_grad_(True)
    b = feat.clone().requires_grad_(True)
    ga = torch.gather(a.unsqueeze(2).expand(2, 4, 5, 5), 3, idx.unsqueeze(1).expand(2, 4, 5, 3))
    gb = gather_knn(b, idx)
    assert torch.equal(ga, gb)
    ga.backward(torch.ones_like(ga))
    gb.backward(torch.ones_like(gb))
    assert torch.allclose(a.grad, b.grad)


def test_gather_knn_error_behaviour():
    from pointmvsnet_b200.functions import dgcnn_ext
    with pytest.raises(RuntimeError):
        dgcnn_ext.gather_knn_forward(torch.zeros(1, 2, 3), torch.zeros(1, 3, 2, dtype=torch.long, device=DEV))
    with pytest.raises(RuntimeError):
        dgcnn_ext.gather_knn_forward(torch.zeros(1, 2, 3, device=DEV), torch.zeros(2, 3, 2, dtype=torch.long, device=DEV))
    # empty input
    out = dgcnn_ext.gather_knn_forward(torch.zeros(1, 2, 0, device=DEV), torch.zeros(1, 0, 4, dtype=torch.long, device=DEV))
    assert tuple(out.shape) == (1, 2, 0, 4)


def test_feature_fetch_known_answer_and_oracle():
    from pointmvsnet_b200.utils.feature_fetcher import FeatureFetcher
    g = load_golden("fetch_known_answer.npz")
    H, W = [int(v) for v in g["hw"]]
    y0, y1, x0, x1 = [int(v) for v in g["crop"]]
    B, V, Cc = g["feats"].shape[:3]
    feats = torch.zeros(B, V, Cc, H, W)
    feats[:, :, :, y0:y1, x0:x1] = g["feats"]
    ff = FeatureFetcher()
    out = ff(feats.to(DEV), g["pts"].to(DEV), g["K"].to(DEV), g["E"].to(DEV)).cpu()
    # the reference's criterion (feature_fetcher.py:97): allclose(gathered, truth, rtol=1e-2)
    # the reference's criterion is allclose(gathered, truth, rtol=1e-2) (feature_fetcher.py:97);
    # features are in [0,1] and the reference run itself is 8e-5 off the analytic value
    assert np.allclose(out[:, 0, :, 0].numpy(), g["truth"].numpy(), rtol=1e-2, atol=5e-4)
    assert torch.allclose(out[:, 0], g["out_view0"], atol=5e-4)
    # random points incl. out-of-image ones (zeros padding) vs the oracle, and E=None
    gen = torch.Generator().manual_seed(5)
    fm = torch.randn(2, 3, 8, 12, 20, generator=gen)
    pts = torch.randn(2, 3, 700, generator=gen) * torch.tensor([60., 60., 30.]).view(1, 3, 1) + \
        torch.tensor([0., 0., 650.]).view(1, 3, 1)
    from pointmvsnet_b200.synthetic import make_cameras
    cams = make_cameras(2, 3, 96, 160, 48)
    K = cams[:, :, 1, :3, :3].clone()
    K[:, :, :2] *= 0.125
    E = cams[:, :, 0, :3, :4].contiguous()
    ref = O.feature_fetch(fm, pts, K, E)
    got = ff(fm.to(DEV), pts.to(DEV), K.to(DEV), E.to(DEV)).cpu()
    assert (ref == 0).any() and (ref != 0).any()
    assert torch.allclose(got, ref, atol=1e-5)
    cam_pts = torch.randn(2, 3, 50, generator=gen) + torch.tensor([0., 0., 5.]).view(1, 3, 1)
    K2 = torch.tensor([[8., 0, 10], [0, 8., 6], [0, 0, 1]]).view(1, 1, 3, 3).expand(2, 3, 3, 3).contiguous()
    assert torch.allclose(ff(fm.to(DEV), cam_pts.to(DEV), K2.to(DEV), None).cpu(),
                          O.feature_fetch(fm, cam_pts, K2, None), atol=1e-5)


def test_feature_fetch_backward_matches_autograd_of_oracle():
    from pointmvsnet_b200.utils.feature_fetcher import FeatureFetcher
    gen = torch.Generator().manual_seed(8)
    fm = torch.randn(1, 2, 4, 9, 11, generator=gen)
    pts = torch.randn(1, 3, 60, generator=gen) + torch.tensor([0., 0., 6.]).view(1, 3, 1)
    K = torch.tensor([[9., 0, 5], [0, 9., 4], [0, 0, 1]]).view(1, 1, 3, 3).expand(1, 2, 3, 3).contiguous()
    a = fm.clone().requires_grad_(True)
    O.feature_fetch(a, pts, K, None).pow(2).sum().backward()
    b = fm.clone().to(DEV).requires_grad_(True)
    FeatureFetcher()(b, pts.to(DEV), K.to(DEV), None).pow(2).sum().backward()
    assert torch.allclose(b.grad.cpu(), a.grad, atol=1e-4)


@pytest.mark.parametrize("shape,ks,k", [((2, 3, 5, 20, 36), 5, 16), ((1, 3, 5, 9, 33), 5, 16),
                                        ((1, 3, 7, 6, 5), 3, 8), ((1, 3, 5, 8, 16), 5, 20),
                                        ((1, 3, 1, 1, 1), 3, 4), ((3, 3, 12, 7, 40), 5, 32)])
def test_knn_bit_exact_vs_oracle(shape, ks, k):
    """Includes ragged tiles, D not a multiple of the depth tile, a single-point cloud and
    tie-heavy inputs (duplicated points): canonical order must match everywhere."""
    from pointmvsnet_b200.utils.torch_utils import get_knn_3d
    gen = torch.Generator().manual_seed(11)
    xyz = torch.randn(*shape, generator=gen)
    xyz[:, :, :, ::3] = xyz[:, :, :, 0:1].clone()  # exact duplicates -> exact ties
    want = O.knn3d(xyz, ks, k)
    got = get_knn_3d(xyz.to(DEV), ks, k)
    assert got.dtype == torch.int64 and tuple(got.shape) == tuple(want.shape)
    assert torch.equal(got.cpu(), want)


def test_knn_golden_reference_clouds():
    """Against get_knn_3d of the reference itself (tests/golden/stages_small.npz): exact on
    tie-free points, equal distance multiset elsewhere (torch.topk tie order is
    implementation defined; rule from SURVEY.md section 8c)."""
    from pointmvsnet_b200.utils.torch_utils import get_knn_3d
    st = load_golden("stages_small.npz")
    for tag in ("it1", "it2"):
        xyz, ref_idx = st[tag + "_xyz"], st[tag + "_knn"]
        B, _, D, H, W = xyz.shape
        got = get_knn_3d(xyz.to(DEV), 5, 16).cpu()
        dist2 = O.knn3d_dist2(xyz, 5)
        srt = torch.sort(dist2, dim=1, stable=True).values
        tie_free = (srt[:, 1:17] != srt[:, :16]).all(dim=1)
        assert torch.equal(got[tie_free], ref_idx[tie_free])
        rc, gc = O.idx_to_candidates(ref_idx, D, H, W), O.idx_to_candidates(got, D, H, W)
        ok = ((rc >= 0) & (gc >= 0)).all(dim=2)
        pr = torch.gather(dist2, 1, rc.clamp(min=0).permute(0, 2, 1)).sort(dim=1).values
        pg = torch.gather(dist2, 1, gc.clamp(min=0).permute(0, 2, 1)).sort(dim=1).values
        assert torch.equal(pr.permute(0, 2, 1)[ok], pg.permute(0, 2, 1)[ok])


def test_knn_errors():
    from pointmvsnet_b200.utils.torch_utils import get_knn_3d
    with pytest.raises(RuntimeError):
        get_knn_3d(torch.zeros(1, 3, 5, 4, 4, device=DEV), 5, 17)
    with pytest.raises(RuntimeError):
        get_knn_3d(torch.zeros(1, 3, 5, 4, 4, device=DEV), 7, 16)


def test_edgeconv_modules_vs_reference_stage_tensors(golden_params):
    from pointmvsnet_b200.networks import EdgeConv, EdgeConvNoC
    st = load_golden("stages_small.npz")
    p = golden_params
    pts = st["ec1_points"]  # the second EdgeConv's output is stored at these points
    for tag in ("it1", "it2"):
        x = st[tag + "_feature"].to(DEV)
        idx = st[tag + "_knn"].to(DEV)
        mods = [EdgeConvNoC(136, 32), EdgeConv(32, 32), EdgeConv(64, 64)]
        with torch.no_grad():
            for l, m in enumerate(mods):
                m.conv1.weight.copy_(p["ec%d_w1" % l]); m.conv2.weight.copy_(p["ec%d_w2" % l])
                m.bn.weight.copy_(p["ec%d_gamma" % l]); m.bn.bias.copy_(p["ec%d_beta" % l])
                m.to(DEV).train()
                x = m(x, idx)
                got = x.cpu()[:, :, pts] if l == 1 else x.cpu()
                ref = st[tag + "_ec%d_out" % l]
                assert torch.allclose(got, ref, atol=2e-5, rtol=1e-4), (tag, l, (got - ref).abs().max())


def test_edgeconv_batch_stats_cover_batch_running_stats_and_eval_mode():
    """B=2 (BN statistics span the batch), running-stat side effect equals nn.BatchNorm2d's,
    eval mode uses running statistics, neighbour order does not matter."""
    from pointmvsnet_b200.networks import EdgeConv
    gen = torch.Generator().manual_seed(21)
    B, Cin, Cout, N, K = 2, 32, 32, 300, 16
    x = torch.randn(B, Cin, N, generator=gen)
    idx = torch.randint(0, N, (B, N, K), generator=gen)
    m = EdgeConv(Cin, Cout)
    with torch.no_grad():
        m.bn.weight.uniform_(0.5, 1.5); m.bn.bias.uniform_(-0.2, 0.2)
    ref_bn = torch.nn.BatchNorm2d(2 * Cout)
    ref_bn.load_state_dict(m.bn.state_dict())
    w1, w2 = m.conv1.weight.detach().clone(), m.conv2.weight.detach().clone()
    want = O.edge_conv(x, idx, w1, w2, m.bn.weight.detach(), m.bn.bias.detach(), True)
    # reference side effect on running stats: feed the same [B,2C,N,K] tensor to nn.BatchNorm2d
    local, edge = O.conv1x1(x, w1), O.conv1x1(x, w2)
    nb = O.gather_knn(edge, idx)
    cen = local.unsqueeze(-1).expand(-1, -1, -1, K)
    ref_bn.train()
    ref_bn(torch.cat([cen, nb - cen], dim=1))
    m = m.to(DEV).train()
    with torch.no_grad():
        got = m(x.to(DEV), idx.to(DEV))
        assert torch.allclose(got.cpu(), want, atol=2e-5, rtol=1e-4)
        assert torch.allclose(m.bn.running_mean.cpu(), ref_bn.running_mean, atol=1e-6)
        assert torch.allclose(m.bn.running_var.cpu(), ref_bn.running_var, atol=1e-6, rtol=1e-5)
        assert int(m.bn.num_batches_tracked) == 1
        perm = torch.randperm(K, generator=gen)
        got_p = m(x.to(DEV), idx[:, :, perm].to(DEV))
        assert torch.allclose(got_p, got, atol=1e-5)
        m.eval()
        ref_bn.eval()
        want_eval = torch.relu(ref_bn(torch.cat([cen, nb - cen], dim=1))).mean(dim=3)
        # our module saw one more train step than ref_bn; align the statistics first
        m.bn.load_state_dict(ref_bn.state_dict())
        got_eval = m(x.to(DEV), idx.to(DEV))
        assert torch.allclose(got_eval.cpu(), want_eval, atol=2e-5, rtol=1e-4)
    with pytest.raises(NotImplementedError):
        m.train()
        m(x.to(DEV), idx.to(DEV))  # grad enabled: forward-only operator refuses


def _run_iteration(pf, cpu, depth, scale, isc, it, params, is_test=True):
    with torch.no_grad():
        res, prob, stg = O.point_flow(depth, isc * cpu["depth_interval"], scale, cpu["pyramids"],
                                      cpu["cam_params_list"], cpu["mean"], cpu["std"], cpu["img_hw"], params,
                                      is_test=is_test, return_stages=True)
        d_gpu, p_gpu = pf(depth.to(DEV), (isc * cpu["depth_interval"]).to(DEV), scale, it,
                          feature_pyramids=[p.to(DEV) for p in cpu["pyramids"]],
                          cam_params_list=cpu["cam_params_list"].to(DEV), mean=cpu["mean"].to(DEV),
                          std=cpu["std"].to(DEV), img_hw=cpu["img_hw"], is_test=is_test)
    return res, prob, stg, d_gpu.cpu(), p_gpu.cpu()


def _check_stages(pf, stg, B):
    dbg = pf.debug_stages()
    S, hs, ws = dbg["S"], dbg["hs"], dbg["ws"]
    r = int(round(S ** 0.5))
    feat = sub_to_ref(dbg["feature"].cpu(), S, B, 5, hs, ws, r)
    assert torch.allclose(feat[:, :112], stg["feature"][:, :112], atol=3e-5, rtol=1e-5)
    assert torch.allclose(feat[:, 112:], stg["feature"][:, 112:], atol=1e-6)
    xyz = sub_to_ref(dbg["xyz"].permute(0, 1, 3, 2).contiguous().cpu(), S, B, 5, hs, ws, r)
    assert torch.allclose(xyz, stg["xyz"], atol=1e-6)
    return dbg


def test_point_flow_iterations_vs_oracle_golden_inputs(golden_weights, golden_params):
    """All three iterations on the inputs of the reference forward (pass_small.npz); each
    iteration starts from the oracle's previous depth so stages see identical inputs."""
    gp = load_golden("pass_small.npz")
    H, W = [int(v) for v in gp["img_hw"]]
    cpu = {"pyramids": [gp["conv1"], gp["conv2"], gp["conv3"]], "cam_params_list": gp["cams"], "mean": gp["mean"],
           "std": gp["std"], "img_hw": (H, W), "depth_interval": gp["cams"][:, 0, 1, 3, 1]}
    pf = _pf(golden_weights)
    depth = gp["coarse_depth"]
    for it, (s, isc) in enumerate(zip((0.125, 0.25, 0.5), (1.0, 0.75, 0.15))):
        res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, depth, s, isc, it, golden_params)
        dbg = _check_stages(pf, stg, 1)
        assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0), (it, (d_gpu - res).abs().max())
        assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0)
        depth = res


def test_point_flow_batch2_train_branch_and_5_views(golden_params):
    """B=2 (BN statistics span the batch, per-sample interval), V=5, and the train branch
    (is_test=False: K scaled by 4*image_scale, one cloud, model.py:162-163,271-293)."""
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    from tests.conftest import load_golden as lg
    cpu = make_pointflow_inputs(64, 128, 5, 2, 48, seed=9)
    cpu["depth_interval"] = cpu["depth_interval"] * torch.tensor([1.0, 0.8])
    pf = _pf(lg("flow_weights.npz"))
    res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, cpu["coarse_depth"], 0.25, 0.75, 1, golden_params)
    _check_stages(pf, stg, 2)
    assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0)
    assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0)
    # train branch: cameras at 1/4 resolution
    cpu_t = make_pointflow_inputs(64, 128, 3, 1, 48, seed=10)
    cpu_t["cam_params_list"][:, :, 1, :2, :3] /= 4.0
    res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu_t, cpu_t["coarse_depth"], 0.25, 0.375, 1, golden_params,
                                                  is_test=False)
    assert pf.debug_stages()["S"] == 1
    assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0)
    assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0)


def test_point_flow_running_stats_and_graph_replay(golden_weights, golden_params):
    """BN running statistics after a 4-sub-cloud iteration equal 4 sequential nn.BatchNorm
    updates; a captured CUDA graph of the whole pass reproduces the eager pass."""
    from pointmvsnet_b200.point_flow import PointFlowPass
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    cpu = make_pointflow_inputs(64, 128, 3, 1, 48, seed=12)
    pf = _pf(golden_weights)
    bn0 = pf.flow_mlp[0][0].bn
    rm0 = bn0.running_mean.clone()
    res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, cpu["coarse_depth"], 0.25, 0.75, 1, golden_params)
    assert int(bn0.num_batches_tracked) == int(golden_weights["flow_mlp.0.0.bn.num_batches_tracked"]) + 4
    assert not torch.equal(bn0.running_mean, rm0)
    # replay the oracle's 4 sub-cloud MLP inputs through nn.BatchNorm1d
    dbg = pf.debug_stages()
    ref = torch.nn.BatchNorm1d(64)
    ref.running_mean.copy_(golden_weights["flow_mlp.0.0.bn.running_mean"])
    ref.running_var.copy_(golden_weights["flow_mlp.0.0.bn.running_var"])
    ref.train()
    edge = dbg["edge"].cpu()  # [S,B,N,224]
    for s_ in range(4):
        ref(O.conv1x1(edge[s_].permute(0, 2, 1).contiguous(), golden_params["mlp0_w"]))
    assert torch.allclose(bn0.running_mean.cpu(), ref.running_mean, atol=1e-5, rtol=1e-4)
    assert torch.allclose(bn0.running_var.cpu(), ref.running_var, atol=1e-5, rtol=1e-4)
    # graph replay == eager
    gpu = {k: ([t.to(DEV) for t in v] if isinstance(v, list) else (v.to(DEV) if torch.is_tensor(v) else v))
           for k, v in cpu.items()}
    with torch.no_grad():
        eager = PointFlowPass(pf).run(gpu["pyramids"], gpu["coarse_depth"], gpu["cam_params_list"],
                                      gpu["depth_interval"], gpu["mean"], gpu["std"], gpu["img_hw"])
        eager = [(d.clone(), p.clone()) for d, p in eager]
        pfp = PointFlowPass(pf).capture(gpu)
        assert pfp.launches_per_pass > 30
        for _ in range(2):
            outs = pfp.replay()
        torch.cuda.synchronize()
    for (de, pe), (dg, pg) in zip(eager, outs):
        assert torch.allclose(de, dg, atol=2e-4) and torch.allclose(pe, pg, atol=2e-5)


def test_full_size_c2_properties_and_oracle_it1():
    """BASELINE config 2 (640x512, 3 src views): iteration 1 against the oracle (about 1 s of
    CPU), later iterations through size-independent properties."""
    from pointmvsnet_b200.point_flow import PointFlow, PointFlowPass
    from pointmvsnet_b200.parallel import state_dict_from_params
    from pointmvsnet_b200.synthetic import make_pointflow_inputs, make_flow_params
    from pointmvsnet_b200.utils.torch_utils import get_knn_3d
    cpu = make_pointflow_inputs(512, 640, 4, 1, 96, seed=0)
    params = make_flow_params(seed=1)
    pf = PointFlow().to(DEV)
    pf.load_state_dict(state_dict_from_params(params, pf.state_dict()))
    pf.train()
    res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, cpu["coarse_depth"], 0.125, 1.0, 0, params)
    _check_stages(pf, stg, 1)
    assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0)
    assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0)
    gpu = {k: ([t.to(DEV) for t in v] if isinstance(v, list) else (v.to(DEV) if torch.is_tensor(v) else v))
           for k, v in cpu.items()}
    with torch.no_grad():
        outs = PointFlowPass(pf).run(gpu["pyramids"], gpu["coarse_depth"], gpu["cam_params_list"],
                                     gpu["depth_interval"], gpu["mean"], gpu["std"], gpu["img_hw"])
    itv = cpu["depth_interval"].item()
    prev = gpu["coarse_depth"]
    for (d, p), s, isc in zip(outs, (0.125, 0.25, 0.5), (1.0, 0.75, 0.15)):
        h, w = int(512 * s), int(640 * s)
        assert tuple(d.shape) == (1, 1, h, w) and tuple(p.shape) == (1, 5, h, w)
        assert torch.isfinite(d).all() and torch.isfinite(p).all()
        assert torch.allclose(p.sum(dim=1), torch.ones(1, h, w, device=DEV), atol=1e-5)  # softmax
        up = torch.nn.functional.interpolate(prev, (h, w), mode="nearest") if prev.shape[2] != h else prev
        assert ((d - up).abs() <= 2 * isc * itv + 1e-3).all()  # expectation stays inside the hypotheses
        prev = d
    # kNN properties on the last iteration's 16 sub-clouds (409 600 points): self first,
    # indices in range, distances ascending
    dbg = pf.debug_stages()
    xyz = dbg["xyz"].reshape(16, 3, 5, 64, 80)
    idx = get_knn_3d(xyz, 5, 16)
    N = 5 * 64 * 80
    assert torch.equal(idx[:, :, 0], torch.arange(N, device=DEV).expand(16, N))
    assert int(idx.min()) >= 0 and int(idx.max()) < N
    assert torch.equal(idx.int(), dbg["idx"].reshape(16, N, 16))


def test_chained_pass_vs_oracle_pass(golden_weights, golden_params):
    """The whole 3-iteration loop (model.py:297-303) through PointFlowPass (in-kernel
    inter_scale multiply) against the oracle's loop.  Errors chain through nearest upsampling,
    re-projection and kNN near-ties, so the bound is statistical (SURVEY.md section 8c):
    mean <= 1e-4 * interval and 99.9th percentile <= 1e-3 * interval at every iteration."""
    from pointmvsnet_b200.point_flow import PointFlowPass
    gp = load_golden("pass_small.npz")
    H, W = [int(v) for v in gp["img_hw"]]
    interval = gp["cams"][:, 0, 1, 3, 1]
    pyr = [gp["conv1"], gp["conv2"], gp["conv3"]]
    want = O.point_flow_pass(gp["coarse_depth"], interval, pyr, gp["cams"], gp["mean"], gp["std"], (H, W),
                             golden_params)
    pf = _pf(golden_weights)
    with torch.no_grad():
        got = PointFlowPass(pf).run([p.to(DEV) for p in pyr], gp["coarse_depth"].to(DEV), gp["cams"].to(DEV),
                                    interval.to(DEV), gp["mean"].to(DEV), gp["std"].to(DEV), (H, W))
    for i, ((dw, pw), (dg, pg), isc) in enumerate(zip(want, got, (1.0, 0.75, 0.15))):
        err = (dg.cpu() - dw).abs().flatten()
        itv = float(interval[0]) * isc
        assert err.mean() <= 1e-4 * itv, (i, err.mean(), itv)
        assert torch.quantile(err, 0.999) <= 1e-3 * itv, (i, torch.quantile(err, 0.999), itv)


@pytest.mark.parametrize("mode,rtol", [(0, 2e-6), (3, 1e-5), (1, 3e-3)])
@pytest.mark.parametrize("cin,cout,rows", [(136, 64, 1000), (224, 64, 25600), (64, 128, 300), (64, 16, 4097), (32, 64, 128)])
def test_linear_pm_modes_vs_fp64(mode, rtol, cin, cout, rows):
    """The per-point contraction in its three arithmetic modes (fp32 SIMT, 3xTF32 and TF32 on
    tcgen05) against an fp64 matmul, with fused input BatchNorm+ReLU and output statistics.
    Error is normalised by |x|.|w| per output element (rtol)."""
    from pointmvsnet_b200 import _lib
    gen = torch.Generator().manual_seed(cin * 1000 + cout)
    x = torch.randn(rows, cin, generator=gen).to(DEV)
    w = (torch.randn(cout, cin, generator=gen) / cin ** 0.5).to(DEV)
    gamma = (1 + 0.1 * torch.randn(cin, generator=gen)).to(DEV)
    beta = (0.1 * torch.randn(cin, generator=gen)).to(DEV)
    xs = x.double()
    in_stats = torch.cat([xs.sum(0), (xs * xs).sum(0)]).contiguous()
    y = torch.empty(rows, cout, device=DEV)
    out_stats = torch.zeros(2 * cout, device=DEV, dtype=torch.float64)
    old = _lib.lib.pmvs_get_gemm_mode()
    try:
        _lib.set_gemm_mode(mode)
        _lib.check(_lib.lib.pmvs_linear_pm(x.data_ptr(), cin, w.data_ptr(), y.data_ptr(), cout, 1, rows, cin, cout,
                                           in_stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), float(rows), 1e-5,
                                           out_stats.data_ptr(), _lib.stream_ptr()))
        torch.cuda.synchronize()
    finally:
        _lib.set_gemm_mode(old)
    mean = xs.mean(0)
    var = xs.var(0, unbiased=False)
    xn = torch.relu((xs - mean) / torch.sqrt(var + 1e-5) * gamma.double() + beta.double())
    want = xn @ w.double().t()
    scale = xn.abs() @ w.double().abs().t()
    err = ((y.double() - want).abs() / scale.clamp(min=1e-6)).max().item()
    assert err < rtol, (mode, cin, cout, err)
    # plain TF32 truncates the operands (biased), so its column sums drift by ~1e-3 relative
    srt = 5e-3 if mode == 1 else 1e-4
    assert torch.allclose(out_stats[:cout], want.sum(0), rtol=srt, atol=srt * scale.sum(0).max().item())
    assert torch.allclose(out_stats[cout:], (want * want).sum(0), rtol=2 * srt + 1e-4)


@pytest.mark.parametrize("gemm_opt", [0, 1, 2])
@pytest.mark.parametrize("cin,cout,groups,rows", [(64, 64, 3, 1000), (136, 64, 2, 25600), (64, 128, 5, 333),
                                                  (64, 16, 4, 4097), (32, 64, 16, 640), (224, 64, 2, 129)])
def test_linear_pm_groups_ragged_tiles_both_tcgen05_kernels(gemm_opt, cin, cout, groups, rows):
    """Several BatchNorm groups per launch (per-group input statistics, per-group output sums), row counts that
    are not multiples of the 128-point tile, for both tensor-core kernels (gemm_tc.cu / gemm_ws.cu with register
    prefetch or cp.async staging), 3xTF32.  cin = 64 also reads x as a slice of wider rows, as the fused iteration
    reads EdgeConv 2's input: 64 columns at offset 32 of the 224-column EdgeConv concat (ldx = 224)."""
    from pointmvsnet_b200 import _lib
    gen = torch.Generator().manual_seed(cin * 7 + cout + groups)
    x = (torch.randn(groups, rows, cin, generator=gen) * (1 + torch.arange(groups).view(-1, 1, 1))).to(DEV)
    w = (torch.randn(cout, cin, generator=gen) / cin ** 0.5).to(DEV)
    gamma = (1 + 0.1 * torch.randn(cin, generator=gen)).to(DEV)
    beta = (0.1 * torch.randn(cin, generator=gen)).to(DEV)
    xs = x.double()
    in_stats = torch.cat([xs.sum(1), (xs * xs).sum(1)], dim=1).contiguous()  # [groups, 2*cin]
    y = torch.full((groups, rows, cout), float("nan"), device=DEV)
    out_stats = torch.zeros(groups, 2 * cout, device=DEV, dtype=torch.float64)
    layouts = [(x, cin, 0)]
    if cin == 64:
        # large finite values around the slice: a column read outside it changes the result
        wide = (1e3 * torch.randn(groups, rows, 224, generator=gen)).to(DEV)
        wide[:, :, 32:96] = x
        layouts.append((wide, 224, 32))
    old = _lib.get_option("gemm")
    try:
        _lib.set_option("gemm", gemm_opt)
        for (buf, ldx, col), use_bn in [(lay, bn) for lay in layouts for bn in (True, False)]:
            out_stats.zero_()
            y.fill_(float("nan"))
            _lib.check(_lib.lib.pmvs_linear_pm(buf.data_ptr() + 4 * col, ldx, w.data_ptr(), y.data_ptr(), cout, groups,
                                               rows, cin, cout, in_stats.data_ptr() if use_bn else None,
                                               gamma.data_ptr() if use_bn else None, beta.data_ptr() if use_bn else None,
                                               float(rows), 1e-5, out_stats.data_ptr(), _lib.stream_ptr()))
            torch.cuda.synchronize()
            if use_bn:
                mean = xs.mean(1, keepdim=True)
                var = xs.var(1, unbiased=False, keepdim=True)
                xn = torch.relu((xs - mean) / torch.sqrt(var + 1e-5) * gamma.double() + beta.double())
            else:
                xn = xs
            want = xn @ w.double().t()
            scale = (xn.abs() @ w.double().abs().t()).clamp(min=1e-6)
            err = ((y.double() - want).abs() / scale).max().item()
            assert err < 1e-5, (gemm_opt, use_bn, ldx, cin, cout, err)
            assert torch.allclose(out_stats[:, :cout], want.sum(1), rtol=1e-4, atol=1e-4 * scale.sum(1).max().item())
            assert torch.allclose(out_stats[:, cout:], (want * want).sum(1), rtol=3e-4)
    finally:
        _lib.set_option("gemm", old)


def test_ragged_shapes_six_views_vs_oracle(golden_params, golden_weights):
    """A C5-like shape in miniature: sub-grid 37 x 50 (odd, not a multiple of any tile), 6 views
    (the shared-memory opt-in path of the fetch kernel), iterations 1 and 2, all stages vs oracle."""
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    cpu = make_pointflow_inputs(296, 400, 6, 1, 96, seed=21)
    pf = _pf(golden_weights)
    depth = cpu["coarse_depth"]
    for it, (s_, isc) in enumerate(zip((0.125, 0.25), (1.0, 0.75))):
        res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, depth, s_, isc, it, golden_params)
        _check_stages(pf, stg, 1)
        assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0), (it, (d_gpu - res).abs().max())
        assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0)
        depth = res


@pytest.mark.parametrize("views", [7, 12])
def test_point_flow_many_views_second_descriptor_pass(views, golden_params, golden_weights):
    """V > 6: more than 32 (hypothesis, view) pairs per pixel, i.e. the second descriptor pass of the fetch
    kernel (lane + 32), up to PMVS_MAX_VIEWS = 12."""
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    cpu = make_pointflow_inputs(64, 128, views, 1, 48, seed=30 + views)
    pf = _pf(golden_weights)
    res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, cpu["coarse_depth"], 0.25, 0.75, 1, golden_params)
    _check_stages(pf, stg, 1)
    assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0)
    assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0)


def test_fetch_zero_padding_with_non_finite_features(golden_params, golden_weights):
    """grid_sample's zeros padding yields exact zeros for out-of-image taps whatever the map holds; the fused
    fetch points such taps at an all-zero texel instead of weighting a real texel by 0 (0 * inf = nan)."""
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    cpu = make_pointflow_inputs(64, 128, 3, 1, 48, seed=41)
    # push the source cameras sideways so that many projections leave the image, and poison texel (0, 0)
    cpu["cam_params_list"][:, 1:, 0, 0, 3] += 120.0
    for lvl in cpu["pyramids"]:
        lvl[:, :, :, 0, 0] = float("inf")
    pf = _pf(golden_weights)
    with torch.no_grad():
        stg_feature, _, _ = O.build_point_features(cpu["coarse_depth"], 0.75 * cpu["depth_interval"], 0.25,
                                                   cpu["pyramids"], cpu["cam_params_list"], cpu["mean"], cpu["std"],
                                                   cpu["img_hw"])
        pf(cpu["coarse_depth"].to(DEV), (0.75 * cpu["depth_interval"]).to(DEV), 0.25, 1,
           feature_pyramids=[p.to(DEV) for p in cpu["pyramids"]], cam_params_list=cpu["cam_params_list"].to(DEV),
           mean=cpu["mean"].to(DEV), std=cpu["std"].to(DEV), img_hw=cpu["img_hw"])
    dbg = pf.debug_stages()
    feat = sub_to_ref(dbg["feature"].cpu(), dbg["S"], 1, 5, dbg["hs"], dbg["ws"], 2)[:, :112]
    want = stg_feature[:, :112]
    finite = torch.isfinite(want)
    assert finite.float().mean() > 0.9 and (~finite).any()
    assert torch.equal(torch.isfinite(feat), finite)
    assert torch.allclose(feat[finite], want[finite], atol=3e-5, rtol=1e-5)


def test_sub_cloud_range_equals_the_same_pixels_of_the_full_iteration(golden_weights):
    """pmvs_flow_shape.sub_begin / sub_count (the unit of the C5 multi-GPU split): processing sub-clouds
    [first, first + count) alone writes exactly the pixels (and probabilities) the full iteration writes there -
    sub-clouds are independent calls in the reference (model.py:236-267) - and leaves the others untouched."""
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    cpu = make_pointflow_inputs(128, 192, 3, 2, 48, seed=23)
    pf = _pf(golden_weights)
    pf.update_running_stats = False
    args = dict(feature_pyramids=[p.to(DEV) for p in cpu["pyramids"]], cam_params_list=cpu["cam_params_list"].to(DEV),
                mean=cpu["mean"].to(DEV), std=cpu["std"].to(DEV), img_hw=cpu["img_hw"])
    with torch.no_grad():
        d1, _ = pf(cpu["coarse_depth"].to(DEV), cpu["depth_interval"].to(DEV), 0.125, 0, **args)
        for scale, isc, it in ((0.25, 0.75, 1), (0.5, 0.15, 2)):
            full_d, full_p = pf(d1, (isc * cpu["depth_interval"]).to(DEV), scale, it, **args)
            full_d, full_p = full_d.clone(), full_p.clone()
            r = int(scale * 8)
            for first, count in ((0, 1), (1, r * r - 1), (r * r - 1, 1)):
                out_d = torch.full_like(full_d, -7.0)
                out_p = torch.full_like(full_p, -7.0)
                pf(d1, (isc * cpu["depth_interval"]).to(DEV), scale, it, out=(out_d, out_p), sub_range=(first, count), **args)
                torch.cuda.synchronize()
                mask = torch.zeros(r, r, dtype=torch.bool)
                mask.view(-1)[first:first + count] = True
                h, w = full_d.shape[-2:]
                pix = mask.to(DEV).repeat(h // r, w // r)  # pixel (Y, X) belongs to sub-cloud (Y % r, X % r)
                # (fp64 atomics make the BatchNorm sums order dependent in the last bit, hence not torch.equal)
                assert torch.allclose(out_d[:, 0][:, pix], full_d[:, 0][:, pix], atol=2e-4, rtol=0)
                assert torch.allclose(out_p[:, :, pix], full_p[:, :, pix], atol=1e-5, rtol=0)
                assert (out_d[:, 0][:, ~pix] == -7.0).all() and (out_p[:, :, ~pix] == -7.0).all()
                assert pf.debug_stages()["S"] == count


def test_oplevel_closure_equals_fused_point_flow(golden_weights):
    """The UNCHANGED-model.py mode: the reference closure's control flow (21 cal_sub_flow calls per pass) over the
    stand-alone operators (FeatureFetcher, get_knn_3d, EdgeConvNoC / EdgeConv kernels; flow_mlp = stock fp32 PyTorch)
    reproduces the fused PointFlow pass on the golden inputs of the reference forward."""
    from pointmvsnet_b200.point_flow import PointFlowPass
    from pointmvsnet_b200.point_flow_oplevel import point_flow_pass_oplevel
    gp = load_golden("pass_small.npz")
    H, W = [int(v) for v in gp["img_hw"]]
    interval = gp["cams"][:, 0, 1, 3, 1].to(DEV)
    pyr = [gp[k].to(DEV) for k in ("conv1", "conv2", "conv3")]
    pf = _pf(golden_weights)
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            fused = PointFlowPass(pf).run(pyr, gp["coarse_depth"].to(DEV), gp["cams"].to(DEV), interval,
                                          gp["mean"].to(DEV), gp["std"].to(DEV), (H, W))
            fused = [(d.clone(), p.clone()) for d, p in fused]
            ops = point_flow_pass_oplevel(pf.flow_edge_conv, pf.flow_mlp, gp["coarse_depth"].to(DEV), interval, pyr,
                                          gp["cams"].to(DEV), gp["mean"].to(DEV), gp["std"].to(DEV), (H, W))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    for i, ((df, pfp), (do, po), isc) in enumerate(zip(fused, ops, (1.0, 0.75, 0.15))):
        err = (df - do).abs().flatten()
        itv = float(interval[0]) * isc
        # chained iterations: the same statistical bound as the fused pass against the oracle
        assert err.mean() <= 1e-4 * itv and torch.quantile(err, 0.999) <= 1e-3 * itv, (i, err.mean(), err.max())
        assert (pfp - po).abs().mean() < 1e-4


def test_alternate_kernel_families_agree(golden_weights, golden_params):
    """Every stage of the fused path exists in two kernel families (pmvs_set_option): the defaults and the
    round-1 / generic kernels that the stand-alone operators and the unusual shapes still use.  Both must match the
    oracle on the same iteration (and therefore each other)."""
    from pointmvsnet_b200 import _lib
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    cpu = make_pointflow_inputs(64, 128, 4, 1, 48, seed=17)
    saved = {k: _lib.get_option(k) for k in ("edge", "knn", "fetch", "gemm")}
    outs = []
    try:
        for opts in (dict(edge=0, knn=0, fetch=0, gemm=0), dict(edge=1, knn=1, fetch=2, gemm=1), dict(saved)):
            for k, v in opts.items():
                _lib.set_option(k, v)
            pf = _pf(golden_weights)
            res, prob, stg, d_gpu, p_gpu = _run_iteration(pf, cpu, cpu["coarse_depth"], 0.25, 0.75, 1, golden_params)
            _check_stages(pf, stg, 1)
            assert torch.allclose(d_gpu, res, atol=5e-4, rtol=0), opts
            assert torch.allclose(p_gpu, prob, atol=5e-5, rtol=0), opts
            outs.append(d_gpu)
    finally:
        for k, v in saved.items():
            _lib.set_option(k, v)
    assert torch.allclose(outs[0], outs[2], atol=2e-4)


def test_coarse_cost_volume_golden_and_oracle():
    """(f-1) plane-sweep fetch + variance: against the cost volume the reference forward fed to
    VolumeConv (every 6th plane, coarse_small.npz; tolerance 2e-5) and against the oracle on a
    larger white-noise case with out-of-image projections.  White-noise features turn the fp32
    rounding of the projected coordinate (a few 1e-5 px at coordinates ~50 px, CPU bmm vs the
    kernel's FMA chain) directly into feature differences, so that case uses 2e-4 (measured:
    2.3e-5 test mode, 7.1e-5 train mode where coordinates are 2x larger, on 0.03 % of the voxels)."""
    from pointmvsnet_b200.cost_volume import build_cost_volume
    from pointmvsnet_b200.synthetic import make_cameras
    g = load_golden("coarse_small.npz")
    cost = build_cost_volume(g["features"].to(DEV), g["cams"].to(DEV), is_test=True).cpu()
    stride = int(g["plane_stride"])
    assert tuple(cost.shape) == (1, 64, 48, 8, 16)
    assert torch.allclose(cost[:, :, ::stride], g["cost_planes"], atol=2e-5, rtol=1e-5)
    gen = torch.Generator().manual_seed(31)
    feats = torch.randn(2, 5, 32, 20, 28, generator=gen)
    cams = make_cameras(2, 5, 160, 224, 96)
    want, _ = O.coarse_cost_volume(feats, cams, is_test=True)
    got = build_cost_volume(feats.to(DEV), cams.to(DEV), is_test=True).cpu()
    assert torch.allclose(got, want, atol=2e-4, rtol=1e-5), (got - want).abs().max()
    assert ((got - want).abs() > 2e-5).float().mean() < 1e-3
    want_t, _ = O.coarse_cost_volume(feats, cams, is_test=False)
    got_t = build_cost_volume(feats.to(DEV), cams.to(DEV), is_test=False).cpu()
    assert torch.allclose(got_t, want_t, atol=2e-4, rtol=1e-5), (got_t - want_t).abs().max()
    assert ((got_t - want_t).abs() > 2e-5).float().mean() < 1e-3


def test_edgeconv_generic_paths_runtime_k_and_simt_fallback():
    """K != 16 (runtime-K gather loop), out_channels 16 (the 16-channel instance of the gather EdgeConv kernels;
    its contraction, cin 16 -> 2 x 16 = 32 columns, runs on the warp-specialised tcgen05 GEMM, gemm_ws.cu, like
    the other shapes here) and a ragged point count."""
    from pointmvsnet_b200.networks import EdgeConv, EdgeConvNoC
    gen = torch.Generator().manual_seed(41)
    for cls, cin, cout, K, concat in ((EdgeConv, 16, 16, 8, True), (EdgeConvNoC, 24, 32, 5, False),
                                      (EdgeConv, 64, 64, 16, True)):
        B, N = 2, 333
        x = torch.randn(B, cin, N, generator=gen)
        idx = torch.randint(0, N, (B, N, K), generator=gen)
        m = cls(cin, cout)
        with torch.no_grad():
            m.bn.weight.uniform_(0.5, 1.5); m.bn.bias.uniform_(-0.2, 0.2)
        want = O.edge_conv(x, idx, m.conv1.weight.detach(), m.conv2.weight.detach(), m.bn.weight.detach(),
                           m.bn.bias.detach(), concat)
        m = m.to(DEV).train()
        with torch.no_grad():
            got = m(x.to(DEV), idx.to(DEV))
        assert torch.allclose(got.cpu(), want, atol=2e-5, rtol=1e-4), (cls.__name__, (got.cpu() - want).abs().max())


def test_point_flow_refuses_eval_mode(golden_weights):
    pf = _pf(golden_weights).eval()
    with pytest.raises(NotImplementedError):
        pf(torch.zeros(1, 1, 8, 16, device=DEV), torch.ones(1, device=DEV), 0.125, 0,
           feature_pyramids=[torch.zeros(1, 3, 16, 32, 64, device=DEV), torch.zeros(1, 3, 32, 16, 32, device=DEV),
                             torch.zeros(1, 3, 64, 8, 16, device=DEV)],
           cam_params_list=torch.zeros(1, 3, 2, 4, 4, device=DEV), mean=torch.zeros(1, 3, device=DEV),
           std=torch.ones(1, 3, device=DEV))


def test_channels_last_image_conv_feeds_point_flow_without_transposes(golden_weights):
    """SURVEY 8 row f1: ``ImageConv(channels_last=True)`` + ``stack_views_channels_last`` hand PointFlow pyramids that
    already are [B,V,h,w,C] in memory.  They are consumed zero-copy (same storage, three launches fewer than with the
    reference's NCHW stack) and give the same depth map, bit for bit, as the NCHW copy of the same values."""
    from pointmvsnet_b200 import _lib
    from pointmvsnet_b200.networks import ImageConv, stack_views_channels_last
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    H, W, V = 128, 160, 3
    cpu = make_pointflow_inputs(H, W, V, 1, 48, seed=5)
    torch.manual_seed(3)
    conv = ImageConv(8).to(DEV).train()
    imgs = torch.randn(1, V, 3, H, W, device=DEV)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False  # compare the two layouts in fp32 (SURVEY 8c: TF32 off on a GPU oracle)
    try:
        with torch.no_grad():
            per_view = [conv(imgs[:, v]) for v in range(V)]  # model.py:137-143: one call per view
            ref_conv = ImageConv(8, channels_last=False).to(DEV).train()
            ref_conv.load_state_dict(conv.state_dict())
            nchw_view = ref_conv(imgs[:, 0])
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    for k in ("conv1", "conv2", "conv3"):
        assert per_view[0][k].is_contiguous(memory_format=torch.channels_last)
        # same layers, another cuDNN algorithm (summation order): 10 stacked convolutions + batch-statistics BN
        assert torch.allclose(per_view[0][k], nchw_view[k], atol=2e-3, rtol=2e-3)
    pyr_cl = stack_views_channels_last(per_view)
    levels = [pyr_cl[k] for k in ("conv1", "conv2", "conv3")]
    pf = _pf(golden_weights)
    pf.update_running_stats = False
    passed = pf.pyramids_to_channels_last(levels)
    for a, b in zip(passed, levels):
        assert a.data_ptr() == b.data_ptr() and a.is_contiguous()  # no copy, no transpose
    args = dict(cam_params_list=cpu["cam_params_list"].to(DEV), mean=cpu["mean"].to(DEV), std=cpu["std"].to(DEV),
                img_hw=cpu["img_hw"])
    depth, interval = cpu["coarse_depth"].to(DEV), cpu["depth_interval"].to(DEV)
    with torch.no_grad():
        pf(depth, interval, 0.125, 0, feature_pyramids=levels, **args)  # workspace + weight upload, not counted
        torch.cuda.synchronize()
        n0 = _lib.lib.pmvs_launch_count()
        d_cl, p_cl = pf(depth, interval, 0.125, 0, feature_pyramids=levels, **args)
        d_cl, p_cl = d_cl.clone(), p_cl.clone()
        n1 = _lib.lib.pmvs_launch_count()
        d_nchw, p_nchw = pf(depth, interval, 0.125, 0, feature_pyramids=[l.contiguous() for l in levels], **args)
        n2 = _lib.lib.pmvs_launch_count()
    assert (n2 - n1) - (n1 - n0) == 3, "the NCHW stack costs exactly the three transposes the producer removes"
    assert torch.equal(d_cl, d_nchw) and torch.equal(p_cl, p_nchw)


def _scatter_reference(gout, idx, N):
    """`for p in range(N*K): grad_in[idx[p]] += grad_out[p]`, fp32, in that order (numpy, per batch and channel)."""
    B, C, _, K = gout.shape
    res = np.zeros((B, C, N), dtype=np.float32)
    g = gout.reshape(B, C, -1)
    flat = idx.reshape(B, -1)
    for b in range(B):
        order = np.argsort(flat[b], kind="stable")  # ascending destination, ascending source position inside
        dest = flat[b][order]
        for c in range(C):
            vals = g[b, c][order]
            acc = np.float32(0)
            prev = -1
            for d, v in zip(dest, vals):
                if d < 0 or d >= N:
                    continue
                if d != prev:
                    if prev >= 0:
                        res[b, c, prev] = acc
                    acc, prev = np.float32(0), d
                acc = np.float32(acc + v)
            if prev >= 0:
                res[b, c, prev] = acc
    return res


@pytest.mark.parametrize("case", ["knn_window", "random", "hot_row"])
def test_gather_knn_backward_deterministic_segmented_reduce(case):
    """SURVEY 8 row f3: the deterministic GatherKNNBackward.  Bit-identical to the sequential CPU scatter in source
    order, identical between runs, and equal to the atomic scatter up to fp32 summation order - for the structured
    lists of get_knn_3d, for arbitrary indices (with out-of-range entries, which are skipped) and for a row that
    collects thousands of contributions (the long-segment path)."""
    from pointmvsnet_b200.functions import dgcnn_ext
    from pointmvsnet_b200.utils.torch_utils import get_knn_3d
    torch.manual_seed(11)
    if case == "knn_window":
        xyz = torch.randn(2, 3, 5, 12, 20, device=DEV)
        idx = get_knn_3d(xyz, 5, knn=16)
        B, N, K, C = 2, 5 * 12 * 20, 16, 5
    elif case == "random":
        B, N, K, C = 2, 333, 7, 4
        idx = torch.randint(-2, N + 2, (B, N, K), device=DEV)
    else:
        B, N, K, C = 1, 700, 8, 3
        idx = torch.randint(0, N, (B, N, K), device=DEV)
        idx[:, :, :6] = 17  # 4 200 contributions to one row
    gout = torch.randn(B, C, N, K, device=DEV) * 3
    a = dgcnn_ext.gather_knn_backward(gout, idx)
    b = dgcnn_ext.gather_knn_backward(gout, idx)
    atomic = dgcnn_ext.gather_knn_backward(gout, idx, deterministic=False)
    assert torch.equal(a, b)
    ref = _scatter_reference(gout.cpu().numpy(), idx.cpu().numpy(), N)
    assert np.array_equal(a.cpu().numpy(), ref)
    # the atomic scatter adds in arrival order: rows that collect > 1 000 contributions (the clamped aliases of the
    # out-of-grid picks, the hot row) differ from any fixed order by ~sqrt(n) * |sum| * 2^-24
    assert torch.allclose(a, atomic, rtol=1e-5, atol=2e-3)
