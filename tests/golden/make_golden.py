"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference modules are imported from /root/reference (read-only; bytecode writing
disabled).  Inputs come from scsfm.synth (seeded) and from `det_weights` below
(numpy MT19937 keyed by parameter name, so the oracle/CUDA tests can rebuild the same
weights without torch's RNG).  Outputs are stored as float32 .npz files.
"""
import os
import sys
import zlib

import numpy as np

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "sc-sfmlearner-release_b200"))
sys.path.insert(0, HERE)

import torch  # noqa: E402

from golden_util import det_weights, det_image  # noqa: E402


def _load_reference():
    import importlib
    sys.path.insert(0, "/root/reference")
    mods = {n: importlib.import_module(n) for n in ("inverse_warp", "loss_functions", "models")}
    sys.path.remove("/root/reference")
    return mods


def np32(t):
    return t.detach().to(torch.float32).cpu().numpy()


def golden_warp_loss(ref, out):
    from scsfm import synth
    iw, lf = ref["inverse_warp"], ref["loss_functions"]
    B, H, W = 2, 64, 128
    d = synth.loss_inputs(7, B, H, W, n_ref=2, n_scales=2)
    # larger motion than the synth default so that some points leave the frame
    poses = [p * 3 for p in d["poses"]]
    poses_inv = [p * 3 for p in d["poses_inv"]]
    out["in_tgt_img"] = np32(d["tgt_img"])
    for i, r in enumerate(d["ref_imgs"]):
        out[f"in_ref_img{i}"] = np32(r)
    out["in_K"] = np32(d["intrinsics"])
    for s, t in enumerate(d["tgt_depth"]):
        out[f"in_tgt_depth_s{s}"] = np32(t)
    for i, r in enumerate(d["ref_depths"]):
        for s, t in enumerate(r):
            out[f"in_ref_depth{i}_s{s}"] = np32(t)
    for i in range(2):
        out[f"in_pose{i}"] = np32(poses[i])
        out[f"in_pose_inv{i}"] = np32(poses_inv[i])

    for pm in ("zeros", "border"):
        iw.pixel_coords = None
        # (1) inverse_warp2 maps for pair (tgt <- ref0)
        w, v, pd, cd = iw.inverse_warp2(d["ref_imgs"][0], d["tgt_depth"][0], d["ref_depths"][0][0], poses[0],
                                        d["intrinsics"], pm)
        out[f"{pm}_warped"], out[f"{pm}_valid"] = np32(w), np32(v)
        out[f"{pm}_proj_depth"], out[f"{pm}_comp_depth"] = np32(pd), np32(cd)
        # (2) scalar losses for flag combinations (ssim, mask, auto_mask), 2 scales
        for flags in ((1, 1, 1), (1, 1, 0), (0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1)):
            p, g = lf.compute_photo_and_geometry_loss(d["tgt_img"], d["ref_imgs"], d["intrinsics"], d["tgt_depth"],
                                                      d["ref_depths"], poses, poses_inv, 2, *flags, pm)
            out[f"{pm}_loss_{flags[0]}{flags[1]}{flags[2]}"] = np.array([float(p), float(g)], np.float32)
        # (3) gradients of 1*photo + 0.5*geo + 0.1*smooth, flags (1,1,0) and (1,1,1), 2 scales
        for flags in ((1, 1, 0), (1, 1, 1)):
            td = [t.clone().requires_grad_(True) for t in d["tgt_depth"]]
            rd = [[t.clone().requires_grad_(True) for t in r] for r in d["ref_depths"]]
            ps = [t.clone().requires_grad_(True) for t in poses]
            pi = [t.clone().requires_grad_(True) for t in poses_inv]
            p, g = lf.compute_photo_and_geometry_loss(d["tgt_img"], d["ref_imgs"], d["intrinsics"], td, rd, ps, pi,
                                                      2, *flags, pm)
            s = lf.compute_smooth_loss(td, d["tgt_img"], rd, d["ref_imgs"])
            (p + 0.5 * g + 0.1 * s).backward()
            tag = f"{pm}_g{flags[0]}{flags[1]}{flags[2]}"
            out[f"{tag}_smooth"] = np.array([float(s)], np.float32)
            for sidx, t in enumerate(td):
                out[f"{tag}_tgt_depth_s{sidx}"] = np32(t.grad)
            for i, r in enumerate(rd):
                for sidx, t in enumerate(r):
                    out[f"{tag}_ref_depth{i}_s{sidx}"] = np32(t.grad)
            for i in range(2):
                out[f"{tag}_pose{i}"] = np32(ps[i].grad)
                out[f"{tag}_pose_inv{i}"] = np32(pi[i].grad)

    # (4) below-threshold case: tiny image -> masked means are the constant 0
    iw.pixel_coords = None
    t = synth.loss_inputs(11, 1, 32, 48, n_ref=1, n_scales=1)
    p, g = lf.compute_photo_and_geometry_loss(t["tgt_img"], t["ref_imgs"], t["intrinsics"], t["tgt_depth"],
                                              t["ref_depths"], t["poses"], t["poses_inv"], 1, 1, 1, 1, "zeros")
    out["tiny_loss"] = np.array([float(p), float(g)], np.float32)
    out["tiny_smooth"] = np.array([float(lf.compute_smooth_loss(t["tgt_depth"], t["tgt_img"], t["ref_depths"],
                                                                t["ref_imgs"]))], np.float32)

    # (5) pose -> matrix, both rotation modes, and the legacy inverse_warp
    vec = torch.tensor([[0.1, -0.2, 0.3, 0.05, -0.02, 0.03], [-1.0, 0.5, 2.0, 0.7, -1.1, 2.5]])
    out["pose_vec"] = np32(vec)
    out["pose_mat_euler"] = np32(iw.pose_vec2mat(vec, "euler"))
    out["pose_mat_quat"] = np32(iw.pose_vec2mat(vec, "quat"))
    iw.pixel_coords = None
    w, v = iw.inverse_warp(d["ref_imgs"][0], d["tgt_depth"][0][:, 0], poses[0], d["intrinsics"], "euler", "zeros")
    out["legacy_warped"], out["legacy_valid"] = np32(w), v.numpy()

    # (6) compute_errors on a synthetic gt / prediction pair
    g = torch.Generator().manual_seed(3)
    gt = torch.rand(2, 64, 128, generator=g) * 90
    gt[gt < 9] = 0
    pred = (gt * (1 + 0.2 * torch.randn(2, 64, 128, generator=g))).abs() * 0.37 + 0.05
    out["err_gt"], out["err_pred"] = np32(gt), np32(pred)
    out["err_kitti"] = np.array(lf.compute_errors(gt, pred, "kitti"), np.float64)
    out["err_nyu"] = np.array(lf.compute_errors(gt.clamp(max=12), pred, "nyu"), np.float64)


def golden_nets(ref, out):
    models = ref["models"]
    B, H, W = 2, 64, 96
    img1, img2 = det_image("img1", B, H, W), det_image("img2", B, H, W)
    for layers in (18, 50):
        for kind in ("disp", "pose"):
            net = models.DispResNet(layers, False) if kind == "disp" else models.PoseResNet(layers, False)
            sd = net.state_dict()
            net.load_state_dict(det_weights(sd))
            net.train()
            tag = f"{kind}{layers}"
            if kind == "disp":
                outs = net(img1)
                loss = sum(((1.0 / o) * (i + 1)).mean() for i, o in enumerate(outs))
                for s, o in enumerate(outs):
                    out[f"{tag}_out_s{s}"] = np32(o)
            else:
                o = net(img1, img2)
                loss = (o * torch.arange(1, 7, dtype=o.dtype)).sum() * 100
                out[f"{tag}_out"] = np32(o)
            loss.backward()
            out[f"{tag}_loss"] = np.array([float(loss)], np.float64)
            names, norms, heads = [], [], []
            for k, p in net.named_parameters():
                if p.grad is None:
                    continue
                names.append(k)
                norms.append(float(p.grad.double().norm()))
                h = np.zeros(4, np.float32)
                g4 = np32(p.grad.reshape(-1)[:4])
                h[:g4.size] = g4
                heads.append(h)
            out[f"{tag}_grad_names"] = np.array(names)
            out[f"{tag}_grad_norms"] = np.array(norms, np.float64)
            out[f"{tag}_grad_heads"] = np.stack(heads)
            # BN running statistics after one training forward
            sd2 = net.state_dict()
            rk = [k for k in sd2 if k.endswith("running_mean") or k.endswith("running_var")]
            out[f"{tag}_running_names"] = np.array(rk)
            out[f"{tag}_running_norms"] = np.array([float(sd2[k].double().norm()) for k in rk], np.float64)
            # eval-mode output (running statistics, single tensor for DispResNet)
            net.eval()
            with torch.no_grad():
                e = net(img1) if kind == "disp" else net(img1, img2)
            out[f"{tag}_eval_out"] = np32(e)
            out[f"{tag}_keys"] = np.array(list(sd.keys()))
            out[f"{tag}_shapes"] = np.array(["x".join(map(str, v.shape)) for v in sd.values()])


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ref = _load_reference()
    a = {}
    golden_warp_loss(ref, a)
    parts = {}          # by key prefix, so that every file stays under 1 MB (tests/conftest.py merges them)
    for k, v in a.items():
        p = k.split("_")[0]
        parts.setdefault(p if p in ("in", "zeros", "border") else "misc", {})[k] = v
    for p, d in parts.items():
        np.savez_compressed(os.path.join(HERE, "warp_loss_%s.npz" % p), **d)
    b = {}
    golden_nets(ref, b)
    np.savez_compressed(os.path.join(HERE, "nets.npz"), **b)
    for f in ["warp_loss_%s.npz" % p for p in parts] + ["nets.npz"]:
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
