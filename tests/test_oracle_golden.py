"""Pins the CPU oracle (oracle/pointflow_oracle.py) against golden vectors produced
by the reference's own Python (tests/golden/make_golden.py).  CPU only."""
import torch

from oracle import pointflow_oracle as O
from tests.conftest import load_golden


def test_fetch_known_answer():
    """Reference known-answer test, utils/feature_fetcher.py:63-97: a point built to
    project to uv=(60.5, 80.5) fetches features[..., 80, 60] (rtol 1e-2 there)."""
    g = load_golden("fetch_known_answer.npz")
    H, W = [int(v) for v in g["hw"]]
    y0, y1, x0, x1 = [int(v) for v in g["crop"]]
    B, V, C = g["feats"].shape[:3]
    feats = torch.zeros(B, V, C, H, W)
    feats[:, :, :, y0:y1, x0:x1] = g["feats"]
    out = O.feature_fetch(feats, g["pts"], g["K"], g["E"])
    # analytic answer
    assert torch.allclose(out[:, 0, :, 0], g["truth"], rtol=1e-2, atol=1e-3)
    # bit-level agreement with the reference run (same torch build, same ops)
    assert torch.allclose(out[:, 0], g["out_view0"], rtol=0, atol=1e-6)


def test_gather_known_answer():
    """Reference gather test, functions/gather_knn.py:27-56 (fwd == torch.gather, bwd)."""
    g = load_golden("gather_knn.npz")
    assert torch.equal(O.gather_knn(g["feature"], g["index"]), g["out"])
    assert torch.allclose(O.gather_knn_backward(g["grad_out"], g["index"]), g["grad_in"], atol=1e-6)


def _knn_vs_reference(xyz, ref_idx):
    B, _, D, H, W = xyz.shape
    idx, cand, dist2 = O.knn3d(xyz, 5, 16, return_dist=True)
    srt = torch.sort(dist2, dim=1, stable=True).values
    tie_free = (srt[:, 1:17] != srt[:, :16]).all(dim=1)  # [B,N]
    # exact equality where the order is well defined
    assert torch.equal(idx[tie_free], ref_idx[tie_free])
    # elsewhere the picked distance multiset must agree (reference topk tie order is
    # implementation defined); recover distances through candidate ids
    rc = O.idx_to_candidates(ref_idx, D, H, W)
    ok = rc >= 0
    picked = torch.gather(dist2, 1, rc.clamp(min=0).permute(0, 2, 1))
    full = ok.all(dim=2)
    assert torch.equal(torch.sort(picked, dim=1).values.permute(0, 2, 1)[full], srt[:, :16].permute(0, 2, 1)[full])
    return tie_free.float().mean().item()


def test_knn_vs_reference():
    g = load_golden("stages_small.npz")
    for tag in ("it1", "it2"):
        frac = _knn_vs_reference(g[tag + "_xyz"], g[tag + "_knn"])
        assert frac > 0.8  # tiny 8x16 grid: border points tie on the shared zero-pad distance


def test_edgeconv_and_mlp_vs_reference(golden_params):
    g = load_golden("stages_small.npz")
    p = golden_params
    pts = g["ec1_points"]  # the second EdgeConv's output is stored at these points
    for tag in ("it1", "it2"):
        x = g[tag + "_feature"]
        idx = g[tag + "_knn"]  # the reference's own neighbour lists
        outs = []
        for l in range(3):
            x = O.edge_conv(x, idx, p["ec%d_w1" % l], p["ec%d_w2" % l], p["ec%d_gamma" % l],
                            p["ec%d_beta" % l], concat_central=(l > 0))
            got, ref = (x[:, :, pts] if l == 1 else x), g[tag + "_ec%d_out" % l]
            assert torch.allclose(got, ref, rtol=1e-4, atol=1e-4), (tag, l, (got - ref).abs().max())
            outs.append(x)
        y = O.flow_mlp(torch.cat(outs, dim=1), p)
        assert torch.allclose(y, g[tag + "_mlp_out"], rtol=1e-4, atol=2e-4), (y - g[tag + "_mlp_out"]).abs().max()


def test_point_flow_pass_vs_reference(golden_params):
    """Oracle iteration loop == the reference forward's flow1..3 given the same pyramids
    and coarse depth (model.py:297-303)."""
    g = load_golden("pass_small.npz")
    H, W = [int(v) for v in g["img_hw"]]
    interval = g["cams"][:, 0, 1, 3, 1]
    # The reference's topk tie order is implementation defined and this 8x16 grid is
    # border-dominated (2.3 % of points tie exactly at rank 16/17 on the shared zero-pad
    # distance), so the loop is replayed with the reference's own neighbour lists; the
    # kNN itself is pinned by test_knn_vs_reference.
    calls = iter(g["knn_all"].long())
    outs = O.point_flow_pass(g["coarse_depth"], interval, [g["conv1"], g["conv2"], g["conv3"]], g["cams"],
                             g["mean"], g["std"], (H, W), golden_params, knn_fn=lambda xyz: next(calls))
    for i, (depth, prob) in enumerate(outs):
        rd, rp = g["flow%d" % (i + 1)], g["flow%d_prob" % (i + 1)]
        err = (depth - rd).abs()
        assert err.max() < 2e-3, (i, err.max())  # mm, depths are ~650 mm (fp32 ulp 6e-5)
        assert (prob - rp).abs().max() < 1e-4


def test_coarse_cost_volume_vs_reference():
    """(f-1) plane-sweep fetch + variance of the coarse stage, model.py:54-113."""
    g = load_golden("coarse_small.npz")
    cost, depths = O.coarse_cost_volume(g["features"], g["cams"], is_test=True)
    stride = int(g["plane_stride"])
    assert torch.allclose(cost[:, :, ::stride], g["cost_planes"], atol=1e-6)
    assert depths.shape[1] == 48
