"""Evaluation / side-channel rows of SURVEY.md section 8(f): the device `compute_errors` (masked per-image median select +
metrics, reference loss_functions.py:163-205) and the validation loops of train.py (reference train.py:302-423) against the
oracle.  Needs a GPU."""
import argparse

import numpy as np
import pytest
import torch

from golden_util import det_weights

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _gt_pred(seed, B, H, W, quantised):
    g = torch.Generator().manual_seed(seed)
    gt = 0.05 + 90 * torch.rand(B, H, W, generator=g) ** 2          # some pixels below 0.1, some above 80
    pred = gt * (0.6 + 0.8 * torch.rand(B, H, W, generator=g)) * 0.37
    pred[:, ::7, ::5] = 1e-5                                          # clamped to 1e-3
    if quantised:                                                     # heavy ties around the medians
        gt, pred = (gt * 4).round() / 4, (pred * 8).round() / 8
    gt[0, :, : W // 2] = 0                                            # an image with a different (odd / even) valid count
    return gt, pred


@pytest.mark.parametrize("shape", [(3, 37, 61), (2, 96, 160), (4, 256, 832)])
@pytest.mark.parametrize("quantised", [False, True])
@pytest.mark.parametrize("dataset", ["kitti", "nyu"])
def test_compute_errors_kernel_vs_oracle(shape, quantised, dataset):
    import loss_functions as lf
    from oracle import losses as OL
    from scsfm import loss_ops
    B, H, W = shape
    gt, pred = _gt_pred(11, B, H, W, quantised)
    if dataset == "nyu":
        gt = gt.clamp(max=12)
    want = OL.compute_errors(gt, pred, dataset)
    got = lf.compute_errors(gt.to(DEV), pred.to(DEV), dataset)
    np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-7)
    # the medians themselves are exact (bit-identical to torch.median = lower median of the masked values)
    ya, yb, xa, xb, cap = ((0.40810811, 0.99189189, 0.03594771, 0.96405229, 80) if dataset == "kitti" else
                           (0.09375, 0.98125, 0.0640625, 0.9390625, 10))
    per = loss_ops.compute_errors(gt.to(DEV), pred.to(DEV), int(ya * H), int(yb * H), int(xa * W), int(xb * W), float(cap)).cpu()
    crop = torch.zeros(H, W, dtype=torch.bool)
    crop[int(ya * H):int(yb * H), int(xa * W):int(xb * W)] = True
    for b in range(B):
        sel = (gt[b] > 0.1) & (gt[b] < cap) & crop
        assert float(per[b, 6]) == float(torch.median(gt[b][sel]))
        assert float(per[b, 7]) == float(torch.median(pred[b][sel].clamp(1e-3, cap)))


def test_compute_errors_rejects_bad_input_and_flags_empty_masks():
    import loss_functions as lf
    with pytest.raises(ValueError):
        lf.compute_errors(torch.ones(1, 8, 8, device=DEV), torch.ones(1, 8, 8, device=DEV), "cityscapes")
    out = lf.compute_errors(torch.zeros(2, 32, 32, device=DEV), torch.ones(2, 32, 32, device=DEV), "kitti")     # nothing valid
    assert all(np.isnan(v) for v in out)


def _nets(mode):
    import models
    from oracle import nets as N
    disp, pose, odisp, opose = models.DispResNet(18, False), models.PoseResNet(18, False), N.DispResNet(18), N.PoseResNet(18)
    for a, b in ((disp, odisp), (pose, opose)):
        sd = det_weights(b.state_dict())
        a.load_state_dict(sd)
        b.load_state_dict(sd)
    return disp.to(DEV).set_conv_mode(mode), pose.to(DEV).set_conv_mode(mode), odisp.eval(), opose.eval()


@pytest.mark.parametrize("mode", ["fp32", "tf32x3"])
def test_validate_without_gt_matches_the_oracle(mode):
    """train.py:302-362 -- eval-mode networks (running statistics), photometric / geometry / smoothness losses without auto-mask."""
    import train as T
    from oracle import losses as OL
    from scsfm import synth
    disp, pose, odisp, opose = _nets(mode)
    args = argparse.Namespace(num_scales=1, with_ssim=1, with_mask=1, padding_mode="zeros")
    loader = T.SyntheticLoader(2, 2, 128, 160, 2, "kitti", 31)
    got, names = T.validate_without_gt(args, loader, disp, pose, torch.device(DEV))
    assert names == ["Total loss", "Photo loss", "Smooth loss", "Consistency loss"]
    want = torch.zeros(4, dtype=torch.float64)
    with torch.no_grad():
        for i in range(2):
            tgt, refs, K = synth.triplet(31 + i, 2, 128, 160, 2, "kitti")
            td = [1 / odisp(tgt)]
            rd = [[1 / odisp(r)] for r in refs]
            ps, pi = [opose(tgt, r) for r in refs], [opose(r, tgt) for r in refs]
            l1, l3 = OL.compute_photo_and_geometry_loss(tgt, refs, K, td, rd, ps, pi, 1, 1, 1, False, "zeros")
            l2 = OL.compute_smooth_loss(td, tgt, rd, refs)
            want += torch.stack([l1, l1, l2, l3]).double()
    want /= 2
    assert float(want[3]) > 0                       # 128x160x2 pixels: the geometry term is above the 10000-pixel threshold
    np.testing.assert_allclose(got, want.tolist(), rtol=2e-4, atol=1e-6)


def test_validate_with_gt_matches_the_oracle():
    """train.py:365-423 -- predicted depth resized to the ground-truth size, then compute_errors."""
    import train as T
    from oracle import losses as OL
    from scsfm import synth
    disp, _, odisp, _ = _nets("fp32")
    g = torch.Generator().manual_seed(5)
    batches = []
    for i in range(2):
        tgt, _, _ = synth.triplet(70 + i, 2, 128, 160, 2, "kitti")
        depth = 0.5 + 40 * torch.rand(2, 100, 140, generator=g)      # ground truth at a different resolution
        batches.append((tgt, depth))
    batches.append((batches[0][0], torch.zeros(2, 0, 0)))            # an empty ground-truth batch is skipped (train.py:386-387)
    args = argparse.Namespace(dataset="kitti")
    got, names = T.validate_with_gt(args, batches, disp, torch.device(DEV))
    assert names == ["abs_diff", "abs_rel", "sq_rel", "a1", "a2", "a3"]
    want = np.zeros(6)
    with torch.no_grad():
        for tgt, depth in batches[:2]:
            out = 1 / odisp(tgt)[:, 0]
            out = torch.nn.functional.interpolate(out.unsqueeze(1), [100, 140]).squeeze(1)
            want += np.array(OL.compute_errors(depth, out, "kitti"))
    np.testing.assert_allclose(got, want / 2, rtol=2e-3, atol=1e-6)


@pytest.mark.parametrize("gpu_augment", [0, 1])
def test_train_entry_end_to_end_on_synthetic_data(tmp_path, gpu_augment):
    """`python train.py synthetic ...` with the reference's flags: two epochs of three iterations (CUDA-graph step, async logging:
    one read-back per print interval), validation after every epoch, checkpoints and the reference's log files
    (train.py:219-232,270-290; utils.py:57-66).  gpu_augment = 1: uint8 frames through the device-side transforms."""
    import csv
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "sc-sfmlearner-release_b200", "train.py"), "synthetic", "--name", "e2e", "--epochs", "2",
           "--epoch-size", "3", "-b", "2", "--synthetic-size", "128", "160", "--resnet-layers", "18", "--num-scales", "1", "-s", "0.1", "-c", "0.5",
           "--sequence-length", "3", "--with-ssim", "1", "--with-mask", "1", "--with-auto-mask", "1", "--with-pretrain", "0", "--print-freq", "2",
           "--gpu-augment", str(gpu_augment)]
    out = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert " * epoch 1 train loss" in out.stdout
    runs = os.listdir(tmp_path / "checkpoints" / "e2e")
    assert len(runs) == 1
    d = tmp_path / "checkpoints" / "e2e" / runs[0]
    files = set(os.listdir(d))
    assert {"dispnet_checkpoint.pth.tar", "exp_pose_checkpoint.pth.tar", "dispnet_model_best.pth.tar", "exp_pose_model_best.pth.tar",
            "progress_log_summary.csv", "progress_log_full.csv"} <= files
    full = list(csv.reader(open(d / "progress_log_full.csv"), delimiter="\t"))
    assert full[0] == ["train_loss", "photo_loss", "smooth_loss", "geometry_consistency_loss"] and len(full) == 1 + 2 * 3
    assert all(np.isfinite(float(v)) for row in full[1:] for v in row)
    summary = list(csv.reader(open(d / "progress_log_summary.csv"), delimiter="\t"))
    assert summary[0] == ["train_loss", "validation_loss"] and len(summary) == 3
    ck = torch.load(d / "dispnet_checkpoint.pth.tar")
    assert ck["epoch"] == 2 and "encoder.encoder.conv1.weight" in ck["state_dict"]


@pytest.mark.parametrize("gpu_augment", [0, 1])
def test_train_entry_on_a_dataset_on_disk(tmp_path, gpu_augment):
    """`python train.py DIR ...` on a tiny JPEG dataset in the reference's folder layout, with dataset classes of the
    reference's interface (the test doubles under tests/reference_loaders) on PYTHONPATH as train.py expects: --gpu-augment 0 =
    the host transform chain in the loader, 1 = uint8 frames + the device-side transforms; training epoch, validation,
    checkpoints."""
    import os
    import subprocess
    import sys
    from helpers import make_disk_dataset, reference_loader_env
    env = reference_loader_env()
    data = make_disk_dataset(str(tmp_path / "data"))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "sc-sfmlearner-release_b200", "train.py"), data, "--name", "disk", "--epochs", "1",
           "--epoch-size", "2", "-b", "2", "-j", "0", "--resnet-layers", "18", "--num-scales", "1", "-s", "0.1", "-c", "0.5",
           "--sequence-length", "3", "--with-ssim", "1", "--with-mask", "1", "--with-auto-mask", "1", "--with-pretrain", "0",
           "--print-freq", "1", "--gpu-augment", str(gpu_augment)]
    out = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    assert " * epoch 0 train loss" in out.stdout or "train loss" in out.stdout, out.stdout[-2000:]
    runs = os.listdir(tmp_path / "checkpoints" / "disk")
    d = tmp_path / "checkpoints" / "disk" / runs[0]
    assert {"dispnet_checkpoint.pth.tar", "exp_pose_checkpoint.pth.tar", "progress_log_full.csv"} <= set(os.listdir(d))
    import csv
    full = list(csv.reader(open(d / "progress_log_full.csv"), delimiter="\t"))
    assert len(full) == 1 + 2 and all(np.isfinite(float(v)) for row in full[1:] for v in row)
