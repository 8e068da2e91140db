"""The U-Net oracle restatement vs outputs of the real reference (tests/golden/unet_*.npz,
written by oracle/make_golden.py from /root/reference/model.py)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import unet_torch

CASES = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "unet_*.npz")))


def _load(path):
    z = np.load(path)
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd::")}
    return z, sd


def _stored_part(z, name, full):
    """The elements of ``full`` that the golden file keeps for gradient ``name``: all of them, or every
    ``stride::<name>``-th element of the flattened tensor where the file stores a strided sample (keeps it under 1 MB)."""
    key = "stride::" + name
    return full.ravel()[::int(z[key])] if key in z.files else full


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_forward_matches_reference(path):
    z, sd = _load(path)
    x = torch.from_numpy(z["x"])
    out = unet_torch.unet_forward(sd, x, torch.float64, per_clip_bn=False).numpy()
    assert out.shape == z["out_batch"].shape
    assert rel_l2(out, z["out_batch"]) < 1e-12
    outc = unet_torch.unet_forward(sd, x, torch.float64, per_clip_bn=True).numpy()
    assert rel_l2(outc, z["out_clip"]) < 1e-12


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_fp32_path_close_to_fp64(path):
    z, sd = _load(path)
    x = torch.from_numpy(z["x"])
    out = unet_torch.unet_forward(sd, x, torch.float32).double().numpy()
    assert rel_l2(out, z["out_batch"]) < 2e-5


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_loss_matches_reference(path):
    z, sd = _load(path)
    out = torch.from_numpy(z["out_batch"])
    tgt = torch.stack([torch.from_numpy(z["x"]), torch.from_numpy(z["phi"])], 1)
    loss, ang, mag = unet_torch.phase_loss(out, tgt)
    assert abs(loss.item() - float(z["loss"])) < 1e-12
    assert abs(ang.item() - float(z["ang_loss"])) < 1e-12
    assert abs(mag.item() - float(z["mag_loss"])) < 1e-12


def test_state_dict_keys_match_reference():
    z, sd = _load(CASES[0])
    mine = unet_torch.random_state_dict(sd["model.0.weight"].shape[1])
    assert set(mine) == set(sd)
    for k in sd:
        assert tuple(mine[k].shape) == tuple(sd[k].shape), k


def test_time_axis_rule():
    """T must be a multiple of 8 and >= 24 (SURVEY.md section 0): the skip concat of
    model.py:113 fails otherwise."""
    sd = unet_torch.random_state_dict(4)
    for T in (24, 32, 120, 136):
        assert unet_torch.unet_forward(sd, torch.randn(1, 4, T)).shape == (1, 8, T)
    for T in (26, 28, 130):
        with pytest.raises(RuntimeError):
            unet_torch.unet_forward(sd, torch.randn(1, 4, T))


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_gradients_match_reference(path):
    """loss.backward() of the reference (train.py:61) vs autograd through the restatement."""
    z, sd = _load(path)
    tgt = torch.stack([torch.from_numpy(z["x"]), torch.from_numpy(z["phi"])], 1)
    loss, ang, mag, grads = unet_torch.loss_and_grads(sd, torch.from_numpy(z["x"]), tgt)
    assert abs(loss - float(z["loss"])) < 1e-12
    for k in z.files:
        if k.startswith("grad::"):
            assert rel_l2(_stored_part(z, k[6:], grads[k[6:]].numpy()), z[k]) < 1e-10, k
