"""Shared helpers for the parity tests."""
import numpy as np
import torch


def t(a, dtype=torch.float32, device="cpu"):
    return torch.from_numpy(np.asarray(a)).to(device=device, dtype=dtype)


def golden_loss_inputs(g, dtype=torch.float32, device="cpu", n_scales=2, requires_grad=False):
    """Rebuild the (tgt_img, ref_imgs, K, tgt_depth, ref_depths, poses, poses_inv) tuple of the golden warp / loss vectors."""
    def leaf(a):
        x = t(a, dtype, device)
        return x.requires_grad_(True) if requires_grad else x
    tgt = t(g["in_tgt_img"], dtype, device)
    refs = [t(g[f"in_ref_img{i}"], dtype, device) for i in range(2)]
    K = t(g["in_K"], dtype, device)
    td = [leaf(g[f"in_tgt_depth_s{s}"]) for s in range(n_scales)]
    rd = [[leaf(g[f"in_ref_depth{i}_s{s}"]) for s in range(n_scales)] for i in range(2)]
    ps = [leaf(g[f"in_pose{i}"]) for i in range(2)]
    pi = [leaf(g[f"in_pose_inv{i}"]) for i in range(2)]
    return tgt, refs, K, td, rd, ps, pi


def rel_l2(a, b):
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def frac_within(a, b, tol):
    """Fraction of elements with |a-b| <= tol * max|b|."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    return float(((a - b).abs() <= tol * b.abs().max()).double().mean())


def make_disk_dataset(root, H=128, W=160, scenes=("scene_a", "scene_b", "scene_v"), frames=5, seed=0):
    """A tiny dataset in the layout the reference's SequenceFolder crawls (datasets/sequence_folders.py:13-21): root/<scene>/
    NNNNNNN.jpg + cam.txt, train.txt / val.txt listing the scene folders (the last scene is the validation scene)."""
    import os
    import numpy as np
    from PIL import Image
    g = np.random.default_rng(seed)
    os.makedirs(root, exist_ok=True)
    for s in scenes:
        d = os.path.join(root, s)
        os.makedirs(d, exist_ok=True)
        base = np.kron(g.integers(40, 216, (H // 16 + 1, W // 16 + 2, 3)).astype(np.float32), np.ones((16, 16, 1), np.float32))
        for i in range(frames):
            im = base[:H, 2 * i:2 * i + W] + g.normal(0, 6, (H, W, 3))          # a slow pan: consecutive frames overlap
            Image.fromarray(np.clip(im, 0, 255).astype(np.uint8)).save(os.path.join(d, "%07d.jpg" % i), quality=95)
        np.savetxt(os.path.join(d, "cam.txt"), np.array([[0.58 * W, 0, 0.49 * W], [0, 1.92 * H, 0.47 * H], [0, 0, 1]]))
    with open(os.path.join(root, "train.txt"), "w") as f:
        f.write("".join(s + "\n" for s in scenes[:-1]))
    with open(os.path.join(root, "val.txt"), "w") as f:
        f.write(scenes[-1] + "\n")
    return root


def reference_loader_env():
    """Environment for a subprocess in which host-side loaders with the reference's interface (datasets/*.py,
    custom_transforms.py: the test doubles under tests/reference_loaders) are importable from PYTHONPATH, as train.py expects
    for real datasets."""
    import os
    loaders = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_loaders")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([loaders] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    return env
