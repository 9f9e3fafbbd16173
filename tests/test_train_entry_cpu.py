"""Host-side behaviour of the train.py entry that needs no GPU: checkpoint files (reference utils.py:57-66 layout, loadable by
the reference's own modules), CLI defaults, ImageNet initialisation from a local file."""
import os
import subprocess
import sys

import pytest
import torch


def test_save_checkpoint_layout_and_roundtrip(tmp_path):
    import models
    import train as T
    disp, pose = models.DispResNet(18, False), models.PoseResNet(18, False)
    T.save_checkpoint(str(tmp_path), {"epoch": 3, "state_dict": disp.state_dict()}, {"epoch": 3, "state_dict": pose.state_dict()}, True)
    files = sorted(os.listdir(tmp_path))
    assert files == ["dispnet_checkpoint.pth.tar", "dispnet_model_best.pth.tar", "exp_pose_checkpoint.pth.tar", "exp_pose_model_best.pth.tar"]
    for prefix, net, cls in (("dispnet", disp, models.DispResNet), ("exp_pose", pose, models.PoseResNet)):
        ck = torch.load(os.path.join(tmp_path, prefix + "_checkpoint.pth.tar"))
        assert ck["epoch"] == 3 and list(ck["state_dict"].keys()) == list(net.state_dict().keys())
        fresh = cls(18, False)
        fresh.load_state_dict(ck["state_dict"])                 # strict
        for k, v in fresh.state_dict().items():
            assert torch.equal(v, net.state_dict()[k]), k
        w = ck["state_dict"]["encoder.encoder.layer1.0.conv1.weight"]
        assert w.is_contiguous() and tuple(w.shape) == (64, 64, 3, 3)      # plain OIHW tensors, not arena views


@pytest.mark.parametrize("layers", [18, 50])
def test_checkpoints_load_into_the_unmodified_reference_modules(tmp_path, layers, golden_nets):
    """The files train.py writes must be usable by the reference's test / inference scripts, i.e. load strictly into the
    reference's own models.DispResNet / PoseResNet.  tests/golden/nets.npz holds, from the unmodified reference modules
    (make_golden.py), their state_dict keys and shapes and their outputs for deterministic weights (one training-mode forward,
    then eval mode with the running statistics it left): the checkpoint must carry exactly those keys and shapes, and loaded
    strictly into the CPU port of the reference networks (oracle/nets.py) reproduce those outputs."""
    import numpy as np
    import models
    import train as T
    from golden_util import det_image, det_weights
    from oracle import nets as N
    disp, pose = models.DispResNet(layers, False), models.PoseResNet(18, False)
    for net in (disp, pose):
        net.load_state_dict(det_weights(net.state_dict()))
    T.save_checkpoint(str(tmp_path), {"epoch": 1, "state_dict": disp.state_dict()}, {"epoch": 1, "state_dict": pose.state_dict()}, False)
    img1, img2 = det_image("img1", 2, 64, 96), det_image("img2", 2, 64, 96)
    for prefix, tag, ref in (("dispnet", "disp%d" % layers, N.DispResNet(layers)), ("exp_pose", "pose18", N.PoseResNet(18))):
        sd = torch.load(os.path.join(tmp_path, prefix + "_checkpoint.pth.tar"))["state_dict"]
        assert list(sd.keys()) == list(golden_nets[tag + "_keys"])
        assert ["x".join(map(str, v.shape)) for v in sd.values()] == list(golden_nets[tag + "_shapes"])
        ref.load_state_dict(sd)                                 # strict
        run = (lambda: ref(img1)) if prefix == "dispnet" else (lambda: ref(img1, img2))
        ref.train()
        with torch.no_grad():
            out = run()
        out, key = (out[0], "_out_s0") if prefix == "dispnet" else (out, "_out")
        np.testing.assert_allclose(out.numpy(), golden_nets[tag + key], rtol=2e-4, atol=2e-5)
        ref.eval()
        with torch.no_grad():
            np.testing.assert_allclose(run().numpy(), golden_nets[tag + "_eval_out"], rtol=2e-4, atol=2e-5)


def test_cli_defaults_and_pretrained_weights(tmp_path, monkeypatch):
    import models
    import train as T
    args = T.parser.parse_args(["synthetic", "--name", "x"])
    assert args.with_pretrain == 0 and args.conv_mode == "tf32x3" and args.batch_size == 4 and args.num_scales == 1
    # the reference's flags are all accepted with their meaning
    args = T.parser.parse_args(["data", "--name", "x", "--resnet-layers", "50", "--num-scales", "1", "-b", "4", "-s", "0.1", "-c", "0.5",
                                "--epoch-size", "1000", "--sequence-length", "3", "--with-ssim", "1", "--with-mask", "1",
                                "--with-auto-mask", "1", "--with-pretrain", "1", "--folder-type", "pair", "--dataset", "nyu"])
    assert args.resnet_layers == 50 and args.with_pretrain == 1 and args.folder_type == "pair"
    # --with-pretrain 1 without a local checkpoint: a clear error naming where to put the file
    monkeypatch.setenv("SCSFM_PRETRAINED_DIR", str(tmp_path))
    monkeypatch.setattr(torch.hub, "get_dir", lambda: str(tmp_path / "hub"))
    with pytest.raises(FileNotFoundError, match="resnet18-\\*.pth"):
        models.DispResNet(18, True)
    # with a local torchvision-format file: encoder initialised from it, multi-image stem = cat([w] * 2, 1) / 2 (resnet_encoder.py:56-57)
    src = models.DispResNet(18, False).encoder.encoder.state_dict()
    torch.save({k: v.clone() for k, v in src.items()}, tmp_path / "resnet18-test.pth")
    d, p = models.DispResNet(18, True), models.PoseResNet(18, True)
    assert torch.equal(d.encoder.encoder.layer2[0].conv1.weight, src["layer2.0.conv1.weight"])
    assert torch.allclose(p.encoder.encoder.conv1.weight, torch.cat([src["conv1.weight"]] * 2, 1) / 2)


def test_real_dataset_loaders_host_side(tmp_path):
    """train.make_loaders on a dataset on disk with dataset classes of the reference's interface on PYTHONPATH (the test doubles
    under tests/reference_loaders): --gpu-augment 0 builds the host transform chain (normalised float tensors come out of the
    loader), --gpu-augment 1 builds the datasets with transform=None and hands uint8 frames [B, n_img, H, W, 3] + intrinsics to
    the device stage (host side checked here, in a clean interpreter; the device stage in tests/test_augment_gpu.py and
    tests/test_eval_gpu.py)."""
    from helpers import make_disk_dataset, reference_loader_env
    env = reference_loader_env()
    data = make_disk_dataset(str(tmp_path / "data"))
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "sc-sfmlearner-release_b200")
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, torch, train as T\n"
            "SF = T._reference_dataset_module('sequence_folders'); assert 'reference_loaders' in SF.__file__, SF.__file__\n"
            "for g in (0, 1):\n"
            "    args = T.parser.parse_args([%r, '--name', 'x', '-b', '2', '-j', '0', '--gpu-augment', str(g)])\n"
            "    class NoGpu(T.GpuAugmentLoader):\n"
            "        def __init__(self, loader, device, train=True): self.loader = loader\n"
            "    T.GpuAugmentLoader = NoGpu\n"
            "    tl, vl = T.make_loaders(args, 0, 1, 'cpu')\n"
            "    if g == 0:\n"
            "        tgt, refs, K, Kinv = next(iter(tl))\n"
            "        print('HOST', tuple(tgt.shape), tgt.dtype, len(refs), tuple(K.shape), float(tgt.mean()) < 3, len(tl))\n"
            "    else:\n"
            "        frames, K = next(iter(tl.loader))\n"
            "        print('RAW', tuple(frames.shape), frames.dtype, tuple(K.shape), K.dtype, len(tl.loader))\n"
            "    if g == 0:\n"
            "        tgt, refs, K, Kinv = next(iter(vl))\n"
            "        print('VAL', tuple(tgt.shape), len(refs), len(vl))\n"
            "    else:\n"
            "        frames, K = next(iter(vl.loader))\n"
            "        print('VALRAW', tuple(frames.shape), frames.dtype, len(vl.loader))\n" % (pkg, data))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = out.stdout.strip().splitlines()
    assert lines[0] == "HOST (2, 3, 128, 160) torch.float32 2 (2, 3, 3) True 3", lines
    assert lines[2] == "RAW (2, 3, 128, 160, 3) torch.uint8 (2, 3, 3) torch.float32 3", lines
    assert lines[1] == "VAL (2, 3, 128, 160) 2 2" and lines[3] == "VALRAW (2, 3, 128, 160, 3) torch.uint8 2", lines
