"""Synthetic inputs and synthetic U-Net weights.  TEST INFRASTRUCTURE ONLY.

The released .pth weights are fetched from GitHub at run time by the reference (mask.py:22-35,
48-52) and there is no network here, so all parity / bench work runs on seeded synthetic
state_dicts that carry the EXACT key layout of
    UNet(n_classes=K, padding=True, depth=5, up_mode="upsample", batch_norm=True, residual=False)
(mask.py:58-65; resunet.py:36-56,73-106,119-136) - 227 tensors including the dead `residual_*`
tensors and the BN `num_batches_tracked` counters - and on seeded CT-like phantoms.
"""
from collections import OrderedDict

import numpy as np
import torch
import torch.nn.functional as F

from . import restate

CH = [64, 128, 256, 512, 1024]


# ------------------------------------------------------------------------------------------------
def phantom(S: int, H: int = 256, W: int = 256, seed: int = 0, sigma: float = 20.0) -> np.ndarray:
    """CT-like int16 volume: air -1000 HU, elliptical body +40 HU, two ellipsoidal lungs -850 HU that
    taper along z, Gaussian noise.  (SURVEY.md Appendix A.)"""
    rng = np.random.default_rng(seed)
    z = np.linspace(-0.8, 0.8, S) if S > 1 else np.zeros(1)
    y = np.linspace(-1, 1, H)
    x = np.linspace(-1, 1, W)
    Z, Y, X = np.meshgrid(z, y, x, indexing="ij")
    vol = np.full((S, H, W), -1000.0)
    vol[(X / 0.85) ** 2 + (Y / 0.65) ** 2 < 1] = 40.0
    for cx in (-0.38, 0.38):
        vol[((X - cx) / 0.28) ** 2 + (Y / 0.42) ** 2 + (Z / 0.9) ** 2 < 1] = -850.0
    vol += rng.normal(0.0, sigma, size=vol.shape)
    return np.rint(vol).astype(np.int16)


def ground_truth(resized: np.ndarray, K: int) -> np.ndarray:
    """Labels on the 256x256 network grid.  K=3: 1 = patient-right lung (low columns), 2 = left
    (README.md:18-28).  K=6: the same lungs cut into lobes 1,2 (left) / 3,4,5 (right) by image row,
    so that a K=6 and a K=3 model trained on this agree on where lung is (needed by the fusion
    rule mask.py:229-230)."""
    S, H, W = resized.shape
    lung = resized < -600
    # lungs only inside the body: drop the air background (connected to the frame)
    body = np.zeros_like(lung)
    for i in range(S):
        from scipy import ndimage
        body[i] = ndimage.binary_fill_holes(resized[i] > -500)
    lung &= body
    cols = np.arange(W)[None, None, :]
    rows = np.arange(H)[None, :, None]
    gt = np.zeros(resized.shape, dtype=np.int64)
    right, left = lung & (cols < W // 2), lung & (cols >= W // 2)
    if K == 3:
        gt[right], gt[left] = 1, 2
    else:
        gt[left & (rows < H // 2)] = 1
        gt[left & (rows >= H // 2)] = 2
        gt[right & (rows < int(H * 0.43))] = 3
        gt[right & (rows >= int(H * 0.43)) & (rows < int(H * 0.57))] = 4
        gt[right & (rows >= int(H * 0.57))] = 5
    return gt


# ------------------------------------------------------------------------------------------------
def schema(K: int):
    """[(key, shape, kind)] in the reference module's registration order."""
    out = []

    def conv(p, co, ci, k, dead=False):
        out.append((p + ".weight", (co, ci, k, k), "dead" if dead else "conv_w"))
        out.append((p + ".bias", (co,), "dead" if dead else "conv_b"))

    def bn(p, c, dead=False):
        tag = "dead_" if dead else ""
        out.append((p + ".weight", (c,), tag + "bn_w"))
        out.append((p + ".bias", (c,), tag + "bn_b"))
        out.append((p + ".running_mean", (c,), tag + "bn_mean"))
        out.append((p + ".running_var", (c,), tag + "bn_var"))
        out.append((p + ".num_batches_tracked", (), "bn_count"))

    def block(p, ci, co):  # resunet.py:73-106
        conv(p + ".residual_input_conv", co, ci, 1, dead=True)
        bn(p + ".residual_batchnorm", co, dead=True)
        conv(p + ".block.0", co, ci, 3)
        bn(p + ".block.2", co)
        conv(p + ".block.3", co, co, 3)
        bn(p + ".block.5", co)

    prev = 1
    for i, c in enumerate(CH):
        block(f"down_path.{i}", prev, c)
        prev = c
    for j, c in enumerate(reversed(CH[:-1])):  # resunet.py:119-136
        p = f"up_path.{j}"
        conv(p + ".residual_input_conv", c, prev, 1, dead=True)
        bn(p + ".residual_batchnorm", c, dead=True)
        conv(p + ".up.1", c, prev, 1)
        block(p + ".conv_block", prev, c)
        prev = c
    conv("last", K, prev, 1)
    return out


def random_state_dict(K: int, seed: int, calibrate_on: np.ndarray = None, head_gain: float = 1.0) -> OrderedDict:
    """He-normal conv weights from numpy's PCG64 (machine-independent), BN affine ~ N(1,0.1)/N(0,0.1),
    BN running stats calibrated by one train-mode pass over `calibrate_on` ((n,256,256) normalised
    fp32 slices; default: 2 phantom slices)."""
    rng = np.random.default_rng(seed)
    sd = OrderedDict()
    for key, shape, kind in schema(K):
        if kind == "bn_count":
            t = torch.zeros((), dtype=torch.int64)
        elif kind in ("conv_w", "dead"):
            if len(shape) == 4:
                fan_in = shape[1] * shape[2] * shape[3]
                t = torch.from_numpy((rng.standard_normal(shape) * np.sqrt(2.0 / fan_in)).astype(np.float32))
            else:
                t = torch.from_numpy((rng.standard_normal(shape) * 0.05).astype(np.float32))
        elif kind == "conv_b":
            t = torch.from_numpy((rng.standard_normal(shape) * 0.05).astype(np.float32))
        elif kind.endswith("bn_w"):
            t = torch.from_numpy((1.0 + 0.1 * rng.standard_normal(shape)).astype(np.float32))
        elif kind.endswith("bn_b"):
            t = torch.from_numpy((0.1 * rng.standard_normal(shape)).astype(np.float32))
        elif kind.endswith("bn_mean"):
            t = torch.zeros(shape, dtype=torch.float32)
        elif kind.endswith("bn_var"):
            t = torch.ones(shape, dtype=torch.float32)
        else:
            raise AssertionError(kind)
        sd[key] = t
    sd["last.weight"] *= head_gain
    if calibrate_on is None:
        vol = phantom(2, seed=seed + 1000)
        tv, _ = restate.preprocess(vol, resolution=[256, 256])
        calibrate_on = restate.normalise(tv).astype(np.float32)
    calibrate_bn(sd, torch.as_tensor(calibrate_on[:, None], dtype=torch.float32))
    return sd


def _upsample2x(x):
    """F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False) from slices and sums, whose backward
    is deterministic on CUDA (F.interpolate's accumulates with atomics)."""
    for d in (2, 3):
        n = x.shape[d]
        prev = torch.cat([x.narrow(d, 0, 1), x.narrow(d, 0, n - 1)], d)
        nxt = torch.cat([x.narrow(d, 1, n - 1), x.narrow(d, n - 1, 1)], d)
        x = torch.stack([0.25 * prev + 0.75 * x, 0.75 * x + 0.25 * nxt], d + 1).flatten(d, d + 1)
    return x


def _forward_train(x, sd, momentum, upsample=None):
    """Same graph as restate.unet_forward but with BN in training mode (updates running stats)."""
    def block(x, p):
        for conv, bn in ((0, 2), (3, 5)):
            x = F.relu(F.conv2d(x, sd[f"{p}.{conv}.weight"], sd[f"{p}.{conv}.bias"], padding=1))
            x = F.batch_norm(x, sd[f"{p}.{bn}.running_mean"], sd[f"{p}.{bn}.running_var"], sd[f"{p}.{bn}.weight"],
                             sd[f"{p}.{bn}.bias"], training=True, momentum=momentum, eps=1e-5)
        return x

    skips = []
    for i in range(5):
        x = block(x, f"down_path.{i}.block")
        if i != 4:
            skips.append(x)
            x = F.avg_pool2d(x, 2)
    for j in range(4):
        up = upsample(x) if upsample else F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False)
        up = F.conv2d(up, sd[f"up_path.{j}.up.1.weight"], sd[f"up_path.{j}.up.1.bias"])
        x = block(torch.cat([up, skips[-j - 1]], 1), f"up_path.{j}.conv_block.block")
    return F.log_softmax(F.conv2d(x, sd["last.weight"], sd["last.bias"]), dim=1)


def calibrate_bn(sd, x):
    """One no-grad train-mode pass with momentum=1 => running stats := this batch's statistics."""
    with torch.no_grad():
        _forward_train(x, sd, momentum=1.0)
    for k in sd:
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.ones((), dtype=torch.int64)


def train_state_dict(K: int, seed: int, steps: int = 60, device: str = None, n_slices: int = 24,
                     batch: int = 4, lr: float = 1e-3, log=None) -> OrderedDict:
    """'Trained-looking' weights: a few Adam steps on phantom ground truth so the label maps are
    clean blobs (~2 components per slice) instead of speckle (SURVEY.md Appendix A).  Harness-only
    use of torch autograd; runs on cuda when available (seconds) else CPU (minutes).  The steps use
    only deterministic kernels, so the same arguments give the same weights on every run."""
    if device is None:
        device = "cuda" if torch.cuda.is_available() else "cpu"
    g = torch.Generator().manual_seed(seed)
    vol = phantom(n_slices, seed=seed + 2000)
    tv, _ = restate.preprocess(vol, resolution=[256, 256])
    x_all = torch.as_tensor(restate.normalise(tv)[:, None], dtype=torch.float32).to(device)
    y_all = torch.as_tensor(ground_truth(tv, K)).to(device)
    sd = random_state_dict(K, seed, calibrate_on=restate.normalise(tv[:2]).astype(np.float32))
    sd = OrderedDict((k, v.to(device)) for k, v in sd.items())
    params = [k for k, _, kind in schema(K) if kind in ("conv_w", "conv_b", "bn_w", "bn_b")]
    for k in params:
        sd[k].requires_grad_(True)
    opt = torch.optim.Adam([sd[k] for k in params], lr=lr)
    cudnn_deterministic = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        for step in range(steps):
            idx = torch.randint(0, n_slices, (batch,), generator=g).to(device)
            logp = _forward_train(x_all[idx], sd, momentum=0.1, upsample=_upsample2x)
            loss = -(logp * F.one_hot(y_all[idx], K).permute(0, 3, 1, 2)).sum(1).mean()   # F.nll_loss without atomics
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()
            if log is not None and (step % 10 == 0 or step == steps - 1):
                log(f"train K={K} step {step} loss {loss.item():.4f}")
    finally:
        torch.backends.cudnn.deterministic = cudnn_deterministic
    for k in params:
        sd[k].requires_grad_(False)
    with torch.no_grad():  # re-calibrate BN on a fixed batch, in eval-compatible form
        _forward_train(x_all[: min(8, n_slices)], sd, momentum=1.0)
    out = OrderedDict((k, v.detach().to("cpu").contiguous()) for k, v in sd.items())
    for k in out:
        if k.endswith("num_batches_tracked"):
            out[k] = torch.tensor(steps + 1, dtype=torch.int64)
    return out


def label_noise_volume(S: int, K: int, seed: int, speckle: float = 5e-4, H: int = 256, W: int = 256) -> np.ndarray:
    """A uint8 label volume shaped like a network output: clean lungs / lobes from the phantom
    geometry plus random single-voxel and small-blob mislabelling - exercises the merge loop,
    largest-component and hole-fill logic of postprocessing without needing a network."""
    rng = np.random.default_rng(seed)
    vol = phantom(S, H, W, seed=seed, sigma=5.0)
    lab = ground_truth(vol.astype(np.int16), K).astype(np.uint8)
    n = int(speckle * lab.size)
    zz, yy, xx = rng.integers(0, S, n), rng.integers(0, H, n), rng.integers(0, W, n)
    lab[zz, yy, xx] = rng.integers(0, K, n).astype(np.uint8)
    for _ in range(max(1, n // 20)):  # small blobs
        z, y, x = rng.integers(0, S), rng.integers(2, H - 2), rng.integers(2, W - 2)
        lab[z, y - 1:y + 2, x - 1:x + 3] = rng.integers(0, K)
    # holes inside lungs
    for _ in range(max(1, S // 4)):
        z, y, x = rng.integers(0, S), rng.integers(90, 166), rng.integers(60, 196)
        lab[z, y:y + 3, x:x + 3] = 0
    return lab
