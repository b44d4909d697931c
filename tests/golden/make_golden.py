#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by running the REFERENCE'S OWN
PYTHON (imported from a PointMVSNet checkout, nothing copied) on CPU.

Run once with the checkout at hand (``python tests/golden/make_golden.py <checkout>``); the
resulting .npz files are committed so that the tests need no reference checkout.
The reference is executed with exactly the three adjustments SURVEY.md
section 8c documents, all applied from outside by monkey-patching:

  1. ``F.grid_sample`` is called with ``align_corners=True`` (PyTorch 1.0.1
     semantics the reference was written for, utils/feature_fetcher.py:51-55);
  2. EdgeConv/EdgeConvNoC take their CUDA branch (networks.py:26-28 / :64-66):
     ``Tensor.is_cuda`` reports True for the duration of their forward and
     ``dgcnn_ext.gather_knn_forward`` is supplied as the expand+gather the real
     extension executes (functions/csrc/gather_knn_kernel.cu:41-44);
  3. the model stays in train mode (test.py:58) so BN uses batch statistics.

Files written:
  flow_weights.npz      hot-path weights of outputs/dtu_wde3/model_pretrained.pth
  fetch_known_answer.npz the reference's own known-answer test (feature_fetcher.py:63-97)
  gather_knn.npz        the reference's own gather test (gather_knn.py:27-56), fwd + bwd
  stages_small.npz      per-stage tensors captured from a real forward (64x128 image),
                        the second EdgeConv's output at the sampled points `ec1_points`
  pass_small.npz        pyramids + coarse depth -> flow1..3, flow{1..3}_prob of that forward
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

if len(sys.argv) != 2:
    sys.exit("usage: make_golden.py <PointMVSNet checkout>")
REF = os.path.abspath(sys.argv[1])
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

# ---- adjustment 2a: the gather the CUDA extension performs -------------------
fake_ext = types.ModuleType("pointmvsnet.functions.dgcnn_ext")


def _gather_fwd(inp, index):
    b, c, n = inp.shape
    k = index.shape[2]
    return inp.unsqueeze(2).expand(b, c, n, n).gather(3, index.unsqueeze(1).expand(b, c, n, k))


def _gather_bwd(grad_output, index):
    b, c, n, k = grad_output.shape
    g = torch.zeros(b, c, n, dtype=grad_output.dtype)
    g.scatter_add_(2, index.unsqueeze(1).expand(b, c, n, k).reshape(b, c, n * k),
                   grad_output.reshape(b, c, n * k))
    return g


fake_ext.gather_knn_forward = _gather_fwd
fake_ext.gather_knn_backward = _gather_bwd
import pointmvsnet.functions  # noqa: E402

sys.modules["pointmvsnet.functions.dgcnn_ext"] = fake_ext
pointmvsnet.functions.dgcnn_ext = fake_ext

import pointmvsnet.utils.feature_fetcher as ref_ff  # noqa: E402
import pointmvsnet.networks as ref_net  # noqa: E402
import pointmvsnet.model as ref_model  # noqa: E402
import pointmvsnet.utils.torch_utils as ref_tu  # noqa: E402
from pointmvsnet.functions.gather_knn import gather_knn as ref_gather_knn  # noqa: E402

# ---- adjustment 1: align_corners=True ---------------------------------------
class _FShim:
    def __getattr__(self, name):
        return getattr(F, name)

    @staticmethod
    def grid_sample(inp, grid, mode="bilinear", padding_mode="zeros"):
        return F.grid_sample(inp, grid, mode=mode, padding_mode=padding_mode, align_corners=True)


ref_ff.F = _FShim()


# ---- adjustment 2b: CUDA branch of EdgeConv* --------------------------------
_orig_is_cuda = torch.Tensor.is_cuda


def _force_cuda_branch(cls):
    orig = cls.forward

    def fwd(self, feature, knn_inds):
        torch.Tensor.is_cuda = property(lambda t: True)
        try:
            return orig(self, feature, knn_inds)
        finally:
            torch.Tensor.is_cuda = _orig_is_cuda

    cls.forward = fwd


_force_cuda_branch(ref_net.EdgeConv)
_force_cuda_branch(ref_net.EdgeConvNoC)

from pointmvsnet_b200.synthetic import make_cameras, DTU_MEAN, DTU_STD  # noqa: E402


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **{k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v))
                                 for k, v in arrays.items()})
    print("wrote", name, "%.1f KB" % (os.path.getsize(path) / 1024))


def load_reference_weights():
    sd = torch.load(os.path.join(REF, "outputs/dtu_wde3/model_pretrained.pth"), map_location="cpu",
                    weights_only=False)["model"]
    return {k[len("module."):] if k.startswith("module.") else k: v for k, v in sd.items()}


def gen_weights(sd):
    keep = {k: v for k, v in sd.items() if k.startswith("flow_edge_conv.") or k.startswith("flow_mlp.")}
    save("flow_weights.npz", **keep)


def gen_fetch_known_answer():
    """The reference's test_feature_fetching (feature_fetcher.py:63-97) on CPU."""
    torch.manual_seed(7)
    B, V, C, H, W, N = 3, 2, 16, 240, 320, 32
    K = torch.tensor([[10, 0, 1], [0, 10, 1], [0, 0, 1]]).float().view(1, 1, 3, 3).expand(B, V, 3, 3).contiguous()
    E = torch.rand(B, V, 3, 4)
    feats = torch.rand(B, V, C, H, W)
    imgpt = torch.tensor([60.5, 80.5, 1.0]).view(1, 1, 3, 1).expand(B, V, 3, N)
    pt = torch.matmul(torch.inverse(K), imgpt) * 200
    pt = torch.matmul(torch.inverse(E[:, :, :, :3]), pt - E[:, :, :, 3].unsqueeze(-1))
    pts = pt[:, 0].contiguous()
    out = ref_ff.FeatureFetcher()(feats, pts, K, E)
    truth = feats[:, :, :, 80, 60][:, 0]
    err = (out[:, 0, :, 0] - truth).abs().max().item()
    print("known-answer max err (align_corners=True):", err)
    assert err < 1e-2
    # features are big; store only a crop that contains every tap of view 0 and
    # let the test rebuild the rest from the seed is fragile -> store fp16-free full view-0/1 crops
    save("fetch_known_answer.npz", K=K, E=E, pts=pts, feats=feats[:, :, :, 78:84, 58:64].contiguous(),
         crop=np.array([78, 84, 58, 64]), hw=np.array([H, W]), out_view0=out[:, 0].contiguous(), truth=truth)


def gen_gather():
    """The reference's test_gather_knn (gather_knn.py:27-56) through GatherKNN.apply."""
    torch.manual_seed(1)
    B, N, C, K = 2, 5, 4, 3
    feat = torch.rand(B, C, N)
    idx = torch.randint(0, N, [B, N, K]).long()
    f = feat.clone().requires_grad_(True)
    out = ref_gather_knn(f, idx)
    gout = torch.rand(B, C, N, K)
    out.backward(gout)
    save("gather_knn.npz", feature=feat, index=idx, out=out, grad_out=gout, grad_in=f.grad)


def gen_forward(sd):
    """A real PointMVSNet.forward (model.py:45-305) on a 64x128, 3-view batch."""
    torch.manual_seed(3)
    H, W, V, D = 64, 128, 3, 48
    net = ref_model.PointMVSNet()
    net.load_state_dict(sd)
    net.train()  # adjustment 3 (test.py:58)
    cams = make_cameras(1, V, H, W, D)
    # keep every projected point well inside the tiny images: shrink the baseline
    batch = {
        "img_list": torch.randn(1, V, 3, H, W),
        "cam_params_list": cams,
        "mean": torch.tensor(DTU_MEAN).view(1, 3),
        "std": torch.tensor(DTU_STD).view(1, 3),
    }
    cap = {"knn": [], "ec": [[], [], []], "mlp": [], "pyr": [], "coarse": [], "cost": []}

    orig_knn = ref_model.get_knn_3d

    def knn_spy(xyz, kernel_size=5, knn=20):
        out = orig_knn(xyz, kernel_size, knn=knn)
        cap["knn"].append((xyz.detach().clone(), out.detach().clone()))
        return out

    ref_model.get_knn_3d = knn_spy
    hooks = []
    for l, m in enumerate(net.flow_edge_conv):
        hooks.append(m.register_forward_hook(
            lambda mod, inp, out, l=l: cap["ec"][l].append((inp[0].detach().clone(), inp[1].detach().clone(),
                                                            out.detach().clone()))))
    hooks.append(net.flow_mlp.register_forward_hook(
        lambda mod, inp, out: cap["mlp"].append((inp[0].detach().clone(), out.detach().clone()))))
    hooks.append(net.flow_img_conv.register_forward_hook(
        lambda mod, inp, out: cap["pyr"].append({k: v.detach().clone() for k, v in out.items()})))
    hooks.append(net.coarse_img_conv.register_forward_hook(
        lambda mod, inp, out: cap["coarse"].append(out["conv3"].detach().clone())))
    hooks.append(net.coarse_vol_conv.register_forward_pre_hook(
        lambda mod, inp: cap["cost"].append(inp[0].detach().clone())))
    with torch.no_grad():
        preds = net(batch, (0.125, 0.25, 0.5), (1.0, 0.75, 0.15), isFlow=True, isTest=True)
    for h in hooks:
        h.remove()
    ref_model.get_knn_3d = orig_knn

    pyr = [torch.stack([p[c] for p in cap["pyr"]], dim=1) for c in ("conv1", "conv2", "conv3")]
    save("pass_small.npz", conv1=pyr[0], conv2=pyr[1], conv3=pyr[2], cams=cams,
         coarse_depth=preds["coarse_depth_map"], mean=batch["mean"], std=batch["std"],
         flow1=preds["flow1"], flow2=preds["flow2"], flow3=preds["flow3"],
         flow1_prob=preds["flow1_prob"], flow2_prob=preds["flow2_prob"], flow3_prob=preds["flow3_prob"],
         img_hw=np.array([H, W]),
         # every get_knn_3d result of the forward (21 calls), so the loop can be replayed
         # with the reference's own (implementation-defined) tie order
         knn_all=torch.stack([k for _, k in cap["knn"]], dim=0).to(torch.int16))
    # coarse stage: per-view conv3 features and every 6th depth plane of the cost volume the
    # reference feeds to VolumeConv (model.py:113-115)
    save("coarse_small.npz", features=torch.stack(cap["coarse"], dim=1), cams=cams,
         cost_planes=cap["cost"][0][:, :, ::6].contiguous(), plane_stride=np.array(6))
    # per-stage tensors: iteration 1 (one cloud) and the first sub-cloud of iteration 2.  The second EdgeConv's
    # output is kept at a fixed eighth of the points (`ec1_points`) so that the file stays under 1 MB; every other
    # tensor is stored whole.
    n_points = cap["knn"][0][1].shape[1]
    pts = np.sort(np.random.default_rng(0).choice(n_points, n_points // 8, replace=False))
    st = {"ec1_points": pts}
    for tag, call in (("it1", 0), ("it2", 1)):
        xyz, idx = cap["knn"][call]
        st[tag + "_xyz"] = xyz
        st[tag + "_knn"] = idx
        for l in range(3):
            fin, kin, fout = cap["ec"][l][call]
            if l == 0:
                st[tag + "_feature"] = fin
            st[tag + "_ec%d_out" % l] = fout[:, :, pts].contiguous() if l == 1 else fout
        st[tag + "_mlp_out"] = cap["mlp"][call][1]
    save("stages_small.npz", **st)
    print("flow1 range", preds["flow1"].min().item(), preds["flow1"].max().item())


if __name__ == "__main__":
    sd = load_reference_weights()
    gen_weights(sd)
    gen_fetch_known_answer()
    gen_gather()
    gen_forward(sd)
