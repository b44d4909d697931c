#!/usr/bin/env python
"""Stage-by-stage parity report (GPU): prints errors of every CUDA stage against the CPU
oracle without asserting.  Used to set / justify the tolerances in tests/test_gpu_parity.py.
Usage: python tests/gpu_report.py [--big]"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pointflow_oracle as O  # noqa: E402
from pointmvsnet_b200 import _lib  # noqa: E402
from pointmvsnet_b200.point_flow import PointFlow, PointFlowPass  # noqa: E402
from pointmvsnet_b200.utils.feature_fetcher import FeatureFetcher  # noqa: E402
from pointmvsnet_b200.utils.torch_utils import get_knn_3d  # noqa: E402
from pointmvsnet_b200.networks import EdgeConv, EdgeConvNoC  # noqa: E402
from pointmvsnet_b200.functions.gather_knn import gather_knn  # noqa: E402
from pointmvsnet_b200.synthetic import make_pointflow_inputs, make_flow_params  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
dev = torch.device("cuda:0")


def gold(name):
    z = np.load(os.path.join(GOLD, name))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def err(name, a, b):
    a = a.detach().float().cpu()
    b = b.detach().float().cpu()
    d = (a - b).abs()
    print("%-34s max_abs %.3e  mean_abs %.3e  ref_max %.3e  max_rel(>1e-3) %.3e" % (
        name, d.max().item(), d.mean().item(), b.abs().max().item(),
        (d / b.abs().clamp(min=1e-3)).max().item()))
    return d


def load_pf(weights):
    pf = PointFlow().to(dev)
    pf.load_reference_state_dict(weights)
    pf.train()
    return pf


def sub_to_ref(t, S, B, M, hs, ws, r):
    """[S,B,N,C] points-major sub-cloud layout -> reference [B,C,M,h,w]."""
    Cc = t.shape[-1]
    x = t.view(r, r, B, M, hs, ws, Cc)  # i, j, b, m, y, x, c
    x = x.permute(2, 6, 3, 4, 0, 5, 1)  # b, c, m, y, i, x, j
    return x.reshape(B, Cc, M, hs * r, ws * r)


def main():
    torch.manual_seed(0)
    w = gold("flow_weights.npz")
    params = O.params_from_state_dict(w)
    print("== gather_knn golden")
    g = gold("gather_knn.npz")
    f = g["feature"].to(dev).requires_grad_(True)
    out = gather_knn(f, g["index"].to(dev))
    err("gather fwd", out, g["out"])
    out.backward(g["grad_out"].to(dev))
    err("gather bwd", f.grad, g["grad_in"])

    print("== fetch known answer")
    g = gold("fetch_known_answer.npz")
    H, W = [int(v) for v in g["hw"]]
    y0, y1, x0, x1 = [int(v) for v in g["crop"]]
    B, V, Cc = g["feats"].shape[:3]
    feats = torch.zeros(B, V, Cc, H, W)
    feats[:, :, :, y0:y1, x0:x1] = g["feats"]
    ff = FeatureFetcher()
    out = ff(feats.to(dev), g["pts"].to(dev), g["K"].to(dev), g["E"].to(dev))
    err("fetch view0 vs reference", out[:, 0], g["out_view0"])
    err("fetch view0 vs analytic", out[:, 0, :, 0], g["truth"])
    # random fetch vs oracle
    inp = make_pointflow_inputs(64, 128, 3, 1, 48, seed=5)
    cams = inp["cam_params_list"]
    K = cams[:, :, 1, :3, :3].clone()
    K[:, :, :2] *= 0.125
    E = cams[:, :, 0, :3, :4].clone()
    fm = torch.randn(1, 3, 8, 8, 16)
    pts = torch.randn(1, 3, 500) * torch.tensor([40., 40., 30.]).view(1, 3, 1) + torch.tensor([0., 0., 650.]).view(1, 3, 1)
    o_ref = O.feature_fetch(fm, pts, K, E)
    o_gpu = ff(fm.to(dev), pts.to(dev), K.to(dev), E.to(dev))
    err("fetch random vs oracle", o_gpu, o_ref)

    print("== knn vs oracle")
    st = gold("stages_small.npz")
    for tag in ("it1", "it2"):
        xyz = st[tag + "_xyz"]
        idx, cand, dist2 = O.knn3d(xyz, 5, 16, return_dist=True)
        got = get_knn_3d(xyz.to(dev), 5, 16).cpu()
        print(tag, "knn exact-equal frac", (got == idx).all(dim=2).float().mean().item(),
              "elements equal", (got == idx).float().mean().item())
    g2 = torch.Generator().manual_seed(11)
    xyz = torch.randn(2, 3, 5, 20, 36, generator=g2)
    for ks, k in ((5, 16), (3, 8), (5, 20)):
        idx = O.knn3d(xyz, ks, k)
        got = get_knn_3d(xyz.to(dev), ks, k).cpu()
        print("random ks=%d k=%d exact" % (ks, k), torch.equal(got, idx))

    print("== EdgeConv modules vs reference stage tensors")
    for tag in ("it1", "it2"):
        x = st[tag + "_feature"].to(dev)
        idx = st[tag + "_knn"].to(dev)
        mods = [EdgeConvNoC(136, 32), EdgeConv(32, 32), EdgeConv(64, 64)]
        with torch.no_grad():
            for l, m in enumerate(mods):
                m.conv1.weight.copy_(params["ec%d_w1" % l]); m.conv2.weight.copy_(params["ec%d_w2" % l])
                m.bn.weight.copy_(params["ec%d_gamma" % l]); m.bn.bias.copy_(params["ec%d_beta" % l])
                m.to(dev).train()
                x = m(x, idx)
                err("%s ec%d" % (tag, l), x[:, :, st["ec1_points"]] if l == 1 else x, st[tag + "_ec%d_out" % l])

    print("== PointFlow iteration stages vs oracle (golden pass inputs)")
    gp = gold("pass_small.npz")
    H, W = [int(v) for v in gp["img_hw"]]
    pf = load_pf(w)
    pyr = [gp["conv1"], gp["conv2"], gp["conv3"]]
    interval = gp["cams"][:, 0, 1, 3, 1]
    depth = gp["coarse_depth"]
    depth_gpu = depth.to(dev)
    pyr_gpu = [p.to(dev) for p in pyr]
    for it, (s, isc) in enumerate(zip((0.125, 0.25, 0.5), (1.0, 0.75, 0.15))):
        with torch.no_grad():
            res, prob, stg = O.point_flow(depth, isc * interval, s, pyr, gp["cams"], gp["mean"], gp["std"], (H, W),
                                          params, return_stages=True)
            d_gpu, p_gpu = pf(depth_gpu, (isc * interval).to(dev), s, it, feature_pyramids=pyr_gpu,
                              cam_params_list=gp["cams"].to(dev), mean=gp["mean"].to(dev), std=gp["std"].to(dev),
                              img_hw=(H, W))
        dbg = pf.debug_stages()
        S, hs, ws_ = dbg["S"], dbg["hs"], dbg["ws"]
        r = int(round(S ** 0.5))
        feat = sub_to_ref(dbg["feature"], S, 1, 5, hs, ws_, r)
        err("it%d feature[0:112] (variance)" % it, feat[:, :112], stg["feature"][:, :112])
        err("it%d feature[112:136] (xyz)" % it, feat[:, 112:], stg["feature"][:, 112:])
        xyz_g = dbg["xyz"].permute(0, 1, 3, 2).contiguous()  # [S,B,N,3]
        err("it%d xyz" % it, sub_to_ref(xyz_g, S, 1, 5, hs, ws_, r), stg["xyz"])
        err("it%d depth" % it, d_gpu, res)
        err("it%d prob" % it, p_gpu, prob)
        err("it%d depth vs reference golden" % it, d_gpu, gp["flow%d" % (it + 1)])
        # chain on identical inputs: feed the oracle result to both
        depth = res
        depth_gpu = res.to(dev)

    if "--big" in sys.argv:
        print("== C2 size timing (eager, no graph)")
        inp = make_pointflow_inputs(512, 640, 4, 1, 96, seed=0, device=dev)
        pfp = PointFlowPass(pf)
        with torch.no_grad():
            for _ in range(3):
                outs = pfp.run(inp["pyramids"], inp["coarse_depth"], inp["cam_params_list"], inp["depth_interval"],
                               inp["mean"], inp["std"], inp["img_hw"])
            torch.cuda.synchronize()
            t0 = time.time()
            n0 = _lib.launch_count()
            for _ in range(10):
                outs = pfp.run(inp["pyramids"], inp["coarse_depth"], inp["cam_params_list"], inp["depth_interval"],
                               inp["mean"], inp["std"], inp["img_hw"])
            torch.cuda.synchronize()
            dt = (time.time() - t0) / 10
        print("eager pass: %.3f ms, %d launches/pass" % (dt * 1e3, (_lib.launch_count() - n0) // 10))
        print("depth range", outs[-1][0].min().item(), outs[-1][0].max().item())
        # iteration 1 vs oracle at full size
        cpu = make_pointflow_inputs(512, 640, 4, 1, 96, seed=0)
        t0 = time.time()
        res, prob = O.point_flow(cpu["coarse_depth"], 1.0 * cpu["depth_interval"], 0.125, cpu["pyramids"],
                                 cpu["cam_params_list"], cpu["mean"], cpu["std"], cpu["img_hw"], params)
        print("oracle it1 %.2f s" % (time.time() - t0))
        with torch.no_grad():
            d_gpu, p_gpu = pf(inp["coarse_depth"], inp["depth_interval"] * 1.0, 0.125, 0,
                              feature_pyramids=inp["pyramids"], cam_params_list=inp["cam_params_list"],
                              mean=inp["mean"], std=inp["std"], img_hw=inp["img_hw"])
        err("C2 it1 depth", d_gpu, res)
        err("C2 it1 prob", p_gpu, prob)


if __name__ == "__main__":
    main()
