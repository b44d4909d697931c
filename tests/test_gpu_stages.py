"""Stage-by-stage parity of the fused PointFlow iteration (``pmvs_point_flow_iter``) with the fp64 oracle.

``PointFlow.debug_stages()`` exposes what each stage of the fused iteration wrote.  Every stage is compared
with oracle code (oracle/pointflow_oracle.py, evaluated in fp64) fed with the GPU's OWN input to that stage,
so that a kNN near-tie or an upstream rounding cannot blur the comparison and each kernel answers for its
own rounding only:

  stage (kernel)                        reference, fed with the GPU's input            bound
  neighbour codes (knn3d.cu)            O.knn3d on the GPU xyz, encoded here           bit exact
  decoded / materialised indices        the oracle's clamped linear indices            bit exact
  EdgeConv 0 / 1 / 2 (edge_tile.cu,     O.edge_conv on GPU feature, edge[0:32],        atol 2e-5 + rtol 1e-4
    edgeconv.cu gather path)              edge[32:96]
  MLP output h2 (gemm_ws.cu)            conv-BN-ReLU x 2, conv on GPU edge             |err| / (|x|.|w|) < 1e-5
  flow head (edgeconv.cu)               BN-ReLU-conv-softmax on GPU h2, depth_up+flow  prob 2e-6, depth 1e-4 mm
  BatchNorm running statistics          S sequential nn.BatchNorm updates (fp64)       rtol 1e-5 + atol 1e-6
    (all six layers, momentum 0.3)        on the reference tensors above;
                                          num_batches_tracked grows by S

Configurations (image H x W, 3 views, batch B, image scale -> sub-grid, S sub-clouds) cover exact tiles, ragged
tiles with two clouds per BatchNorm group, sub-grids smaller than the 8 x 4 tile of the EdgeConv kernels (the TMA
box is larger than the tensor), a one-row grid, the ratio-1 iteration, and a shape whose statistics kernel walks
several tiles per CTA across the cloud boundary.  The out-of-grid neighbour picks (bit 15 of the code, fetched
from the clamped, aliased row) are rare in real clouds; the escape-heavy shapes assert a minimum count of them so
that the path provably runs.  The small shapes also run with the generic kNN kernel's code emission
(``knn=0``) and with the gather EdgeConv path and its statistics layout (``edge=0``).

In the larger grids nearly every out-of-grid pick leaves through the depth layers and is clamped to the first or last
row of the cloud; picks off the image edge, whose linear index wraps into another image row, need the small grids.

Each test records its errors with ``record_property`` (visible with ``--junitxml``) as ratios max |err| / bound, so
1.0 is the bound itself.  Largest ratio over all configurations and kernel families, measured on an NVIDIA B200
(1000 W power limit):

  kNN codes, indices ...... bit exact
  EdgeConv 0 / 1 / 2 ...... 0.12 / 0.042 / 0.20
  h2 ...................... 0.57 (normalised error 5.7e-6)
  prob .................... 0.15 (3.0e-7)
  depth ................... 0.31 (3.1e-5 mm: the rounding of depth_up + flow near 650 mm)
  running statistics ...... 0.17

No bound has 10x headroom, so all stay at the starting points above.  The file runs in about 5 s on the B200
host, most of it the fp64 oracle of `walk` on the CPU.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import pointflow_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MOMENTUM = 0.3
SCALE_ISC = {0.125: 1.0, 0.25: 0.75, 0.5: 0.15}  # image scale -> interval scale of that iteration (model.py:297-303)

# id: (image H, W, batch, image scale, seed, minimum number of out-of-grid picks over all sub-clouds)
CASES = {
    "exact": (64, 128, 1, 0.25, 67, 0),       # 8 x 16 sub-grid, S = 4: exact tiles
    "ragged_b2": (72, 104, 2, 0.5, 75, 600),  # 9 x 13, S = 16: ragged tiles, 2 clouds per group (0.45 % escapes)
    "tiny_b2": (16, 24, 2, 0.25, 19, 1000),   # 2 x 3, S = 4: sub-grid smaller than the tile (51 % escapes)
    "row": (8, 40, 1, 0.5, 11, 1600),         # 1 x 5, S = 16: one-row grid (52 % escapes)
    "single": (24, 40, 1, 0.125, 27, 80),     # 3 x 5, S = 1: ratio-1 iteration (15 % escapes)
    "walk": (192, 320, 2, 0.5, 195, 0),       # 24 x 40, S = 16: several tiles per statistics CTA
}
FAMILIES = {"default": {}, "knn_emit": {"knn": 0, "edge": 1}, "gather": {"edge": 0}}

TOL_EDGE = (2e-5, 1e-4)  # atol, rtol
TOL_H2 = 1e-5
TOL_PROB = 2e-6
TOL_DEPTH = 1e-4
TOL_RUN = (1e-6, 1e-5)


def _pf(weights):
    from pointmvsnet_b200.point_flow import PointFlow
    pf = PointFlow().to(DEV)
    pf.load_reference_state_dict(weights)
    for bn in pf._bn_modules():
        bn.momentum = MOMENTUM  # one value for all six layers: the fused update takes a single momentum
    pf.train()
    return pf


def _cdiv(a, b):
    return -(-a // b)


def run_iteration(weights, cpu, scale, opts, sub_range=None):
    """One fused iteration with kernel options ``opts`` -> dict of CPU tensors: the debug stages, the inputs the
    reference needs besides them, the outputs and the BatchNorm buffers before and after."""
    from pointmvsnet_b200 import _lib
    saved = {k: _lib.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            _lib.set_option(k, v)
        pf = _pf(weights)
        bns = pf._bn_modules()
        before = [(bn.running_mean.cpu().clone(), bn.running_var.cpu().clone(), int(bn.num_batches_tracked))
                  for bn in bns]
        itv = SCALE_ISC[scale] * cpu["depth_interval"]
        with torch.no_grad():
            d, p = pf(cpu["coarse_depth"].to(DEV), itv.to(DEV), scale, 1,
                      feature_pyramids=[t.to(DEV) for t in cpu["pyramids"]],
                      cam_params_list=cpu["cam_params_list"].to(DEV), mean=cpu["mean"].to(DEV),
                      std=cpu["std"].to(DEV), img_hw=cpu["img_hw"], sub_range=sub_range)
        torch.cuda.synchronize()
        dbg = pf.debug_stages()  # reads the options (which buffers hold the neighbour lists): before the restore
        res = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in dbg.items()}
        res["has_codes"] = _lib.get_option("edge") != 0
    finally:
        for k, v in saved.items():
            _lib.set_option(k, v)
    res.update(depth=d.cpu(), prob=p.cpu(), interval=itv, prev_depth=cpu["coarse_depth"], ratio=pf._last[0].ratio,
               sub_begin=sub_range[0] if sub_range else 0, before=before,
               after=[(bn.running_mean.cpu(), bn.running_var.cpu(), int(bn.num_batches_tracked)) for bn in bns])
    return res


def encode_codes(cand, hs, ws):
    """Candidate ids [B,N,16] (d*25 + h*5 + w of the 5x5x5 window) -> the 16-bit neighbour codes of the tile EdgeConv
    kernels: (dd+2)*96 + (dh+2)*12 + (dw+2) for a pick inside the grid, 0x8000 | id outside.  Returns (codes,
    number of picks outside the grid)."""
    N = 5 * hs * ws
    n = torch.arange(N).view(1, N, 1)
    z, y, x = n // (hs * ws), (n // ws) % hs, n % ws
    dd, dh, dw = cand // 25 - 2, (cand % 25) // 5 - 2, cand % 5 - 2
    inside = ((z + dd >= 0) & (z + dd < 5) & (y + dh >= 0) & (y + dh < hs) & (x + dw >= 0) & (x + dw < ws))
    codes = torch.where(inside, (dd + 2) * 96 + (dh + 2) * 12 + (dw + 2), 0x8000 | cand)
    return codes, int((~inside).sum())


def _ratio_err(got, want, atol, rtol):
    """max |got - want| / (atol + rtol |want|): <= 1 is torch.allclose"""
    return ((got.double() - want).abs() / (atol + rtol * want.abs())).max().item()


def _bn_ref(init, channels, dims):
    """nn.BatchNorm in fp64 starting from the weights' buffers"""
    bn = (torch.nn.BatchNorm2d if dims == 2 else torch.nn.BatchNorm1d)(channels, momentum=MOMENTUM).double().train()
    bn.running_mean.copy_(init[0])
    bn.running_var.copy_(init[1])
    return bn


def check_iteration(run, params, min_escape=0):
    """Compares every stage of ``run`` (from run_iteration) with fp64 oracle code; returns the error summary."""
    S, hs, ws = run["S"], run["hs"], run["ws"]
    B = run["feature"].shape[1]
    r, sub_begin = run["ratio"], run["sub_begin"]
    p = {k: v.double() for k, v in params.items()}
    ec_ch, mlp_ch = (32, 64, 128), (64, 64, 16)
    bn_ec = [_bn_ref(run["before"][l], ec_ch[l], 2) for l in range(3)]
    bn_mlp = [_bn_ref(run["before"][3 + l], mlp_ch[l], 1) for l in range(3)]
    err = {"escapes": 0, "edge": [0.0, 0.0, 0.0], "h2": 0.0, "prob": 0.0, "depth": 0.0}
    # depth_up: the previous depth map, nearest-upsampled to the flow grid (O.build_point_features)
    depth_up = run["prev_depth"]
    if depth_up.shape[2:] != run["depth"].shape[2:]:
        depth_up = F.interpolate(depth_up, tuple(run["depth"].shape[2:]), mode="nearest")
    for s in range(S):
        sg = sub_begin + s
        where = "sub-cloud %d" % sg
        # 1. neighbour codes and indices: the oracle's kNN on the GPU's xyz (fp32, as the kernel computes)
        xyz = run["xyz"][s].reshape(B, 3, 5, hs, ws)
        idx, cand, _ = O.knn3d(xyz, 5, 16, return_dist=True)
        codes, esc = encode_codes(cand, hs, ws)
        err["escapes"] += esc
        if run["has_codes"]:
            got = run["cand"][s].to(torch.int64) & 0xFFFF
            bad = (got != codes).any(dim=2)
            assert not bad.any(), (where, "codes differ at (cloud, point)", bad.nonzero()[:8].tolist())
        gidx = run["idx"][s].to(torch.int64)
        assert torch.equal(gidx, idx), (where, "indices differ at", (gidx != idx).any(2).nonzero()[:8].tolist())
        # 2. EdgeConv layers, each on the GPU's input
        edge = run["edge"][s].permute(0, 2, 1).double()  # [B,224,N]
        ins = (run["feature"][s].permute(0, 2, 1).double(), edge[:, 0:32], edge[:, 32:96])
        outs = ((0, 32), (32, 96), (96, 224))
        for l in range(3):
            w1, w2 = p["ec%d_w1" % l], p["ec%d_w2" % l]
            want = O.edge_conv(ins[l], gidx, w1, w2, p["ec%d_gamma" % l], p["ec%d_beta" % l], l > 0)
            got = edge[:, outs[l][0]:outs[l][1]]
            e = _ratio_err(got, want, *TOL_EDGE)
            err["edge"][l] = max(err["edge"][l], e)
            if e > 1:
                d = (got - want).abs() / (TOL_EDGE[0] + TOL_EDGE[1] * want.abs())
                b, c, n = [int(v) for v in (d == d.max()).nonzero()[0]]
                raise AssertionError("%s EdgeConv %d: ratio %.3g at cloud %d channel %d point %d (got %.7g want %.7g)"
                                     % (where, l, e, b, c, n, got[b, c, n], want[b, c, n]))
            # the input of this layer's BatchNorm2d, for the running statistics
            local, nbr = O.conv1x1(ins[l], w1), O.gather_knn(O.conv1x1(ins[l], w2), gidx)
            cen = local.unsqueeze(-1).expand_as(nbr)
            bn_ec[l](torch.cat([cen, nbr - cen], dim=1) if l > 0 else nbr - cen)
        # 3. MLP on the GPU's EdgeConv concat
        x = edge
        for l in range(2):
            y = O.conv1x1(x, p["mlp%d_w" % l])
            bn_mlp[l](y)
            x = torch.relu(O.batch_norm_train(y, p["mlp%d_gamma" % l], p["mlp%d_beta" % l]))
        want = O.conv1x1(x, p["mlp2_w"])
        bn_mlp[2](want)
        scale = O.conv1x1(x.abs(), p["mlp2_w"].abs()).clamp(min=1e-30)
        got = run["h2"][s].permute(0, 2, 1).double()
        e = ((got - want).abs() / scale).max().item()
        err["h2"] = max(err["h2"], e / TOL_H2)
        assert e < TOL_H2, (where, "h2 normalised error", e)
        # 4. flow head on the GPU's h2
        x = torch.relu(O.batch_norm_train(got, p["mlp2_gamma"], p["mlp2_beta"]))
        raw = O.conv1x1(x, p["mlp3_w"]).reshape(B, 5, hs, ws)
        prob = F.softmax(-raw, dim=1)
        length = torch.tensor(O.HYPOTHESES, dtype=torch.float64).view(1, -1, 1, 1) * \
            run["interval"].double().view(-1, 1, 1, 1)
        flow = (prob * length).sum(dim=1, keepdim=True)
        ii, jj = divmod(sg, r)  # pixel (y * r + ii, x * r + jj) belongs to sub-cloud ii * r + jj (model.py:236-255)
        e = _ratio_err(run["prob"][:, :, ii::r, jj::r], prob, TOL_PROB, 0)
        err["prob"] = max(err["prob"], e)
        assert e <= 1, (where, "prob", e * TOL_PROB)
        want_d = depth_up[:, :, ii::r, jj::r].double() + flow
        e = _ratio_err(run["depth"][:, :, ii::r, jj::r], want_d, TOL_DEPTH, 0)
        err["depth"] = max(err["depth"], e)
        assert e <= 1, (where, "depth", e * TOL_DEPTH)
    assert err["escapes"] >= min_escape, ("out-of-grid picks", err["escapes"], min_escape)
    # 5. running statistics of all six BatchNorm layers after S sequential updates
    names = ["flow_edge_conv.%d.bn" % l for l in range(3)] + ["flow_mlp.0.%d.bn" % l for l in range(3)]
    err["run"] = 0.0
    for name, ref, (rm, rv, nbt), (_, _, nbt0) in zip(names, bn_ec + bn_mlp, run["after"], run["before"]):
        assert nbt == nbt0 + S, (name, "num_batches_tracked", nbt, nbt0 + S)
        for what, got, want in (("running_mean", rm, ref.running_mean), ("running_var", rv, ref.running_var)):
            e = _ratio_err(got, want, *TOL_RUN)
            err["run"] = max(err["run"], e)
            assert e <= 1, (name, what, e, (got.double() - want).abs().max().item())
    return err


def _inputs(case):
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    H, W, B, scale, seed, min_escape = CASES[case]
    return make_pointflow_inputs(H, W, 3, B, 48, seed=seed), scale, min_escape


def _record(record_property, err):
    for k, v in err.items():
        record_property(k, v if not isinstance(v, list) else ",".join("%.3g" % x for x in v))


@pytest.mark.parametrize("case,family", [(c, "default") for c in CASES] +
                         [(c, f) for c in ("tiny_b2", "ragged_b2") for f in ("knn_emit", "gather")])
def test_fused_iteration_stages_vs_fp64_oracle(case, family, golden_weights, golden_params, record_property):
    cpu, scale, min_escape = _inputs(case)
    if case == "walk":
        # the launcher's split of the statistics kernel (edge_tile.cu launch_variant): 3 resident CTAs per SM shared
        # equally by the S groups, then the same longest walk with fewer CTAs
        H, W, B = CASES[case][:3]
        r = int(scale * 8)
        hs, ws = int(H * scale) // r, int(W * scale) // r
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        tiles = _cdiv(ws, 8) * _cdiv(hs, 4) * B
        ctas = min(tiles, max(1, 3 * sms // (r * r)))
        ctas = _cdiv(tiles, _cdiv(tiles, ctas))
        record_property("tiles_per_stats_cta", _cdiv(tiles, ctas))
        assert _cdiv(tiles, ctas) >= 2, "the shape no longer makes a statistics CTA walk several tiles"
    run = run_iteration(golden_weights, cpu, scale, FAMILIES[family])
    err = check_iteration(run, golden_params, min_escape)
    _record(record_property, err)


def test_sub_range_stages_and_running_statistics(golden_weights, golden_params, record_property):
    """sub_range=(5, 3) on ragged_b2: the three sub-clouds 5, 6, 7 alone, their pixels, and running statistics equal to
    three sequential updates in that order (num_batches_tracked + 3)."""
    cpu, scale, _ = _inputs("ragged_b2")
    run = run_iteration(golden_weights, cpu, scale, {}, sub_range=(5, 3))
    assert run["S"] == 3
    err = check_iteration(run, golden_params)
    _record(record_property, err)
