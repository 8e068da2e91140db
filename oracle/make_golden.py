"""Generate tests/golden/*.npz by RUNNING THE UNMODIFIED REFERENCE.  Build-container only.

    python oracle/make_golden.py REF_DIR    # REF_DIR: a checkout of LemonATsu/UNet-PhaseGen

What it pins:
  * unet_c{C}_t{T}.npz -- the reference's model.py ``UNetModel(C, 2C, norm_layer=BatchNorm1d)``
    in train mode (the reference never calls .eval()), float64, on seeded input:
    the input, every state_dict entry, the batch-statistics output (train.py:42 semantics),
    the per-clip output (demo.py:33-42 batch-1 loop), and the train.py:45-61 loss with the
    gradient of four weights (the two largest of the C=16 case as every 5th element of the
    flattened tensor, with ``stride::<name>`` = 5, which keeps the file under 1 MB).
    ``matplotlib``/``librosa`` are stubbed only so that model.py:7 (``from utils import ...``)
    resolves; no reference file is copied or modified.
  * stft_*.npz -- the reference has no STFT code of its own (librosa, not installed), so
    these hold outputs of CPU ``torch.stft``/``torch.istft`` configured to librosa's
    semantics, as an independent cross-check of oracle/stft_np.py.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "tests", "golden")


def import_reference_model(ref_dir):
    for name in ("matplotlib", "matplotlib.pyplot", "librosa", "librosa.display"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.use = lambda *a, **k: None
            sys.modules[name] = m
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["librosa"].display = sys.modules["librosa.display"]
    ref_dir = os.path.abspath(ref_dir)
    sys.path.insert(0, ref_dir)
    try:
        for stale in ("model", "utils"):
            sys.modules.pop(stale, None)
        import model as ref_model
    finally:
        sys.path.remove(ref_dir)
    assert os.path.dirname(os.path.abspath(ref_model.__file__)) == ref_dir
    return ref_model


def unet_case(ref_model, C, T, B, seed, grad_stride=1):
    torch.manual_seed(seed)
    net = ref_model.UNetModel(C, 2 * C, norm_layer=nn.BatchNorm1d).double()
    net.train()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, nn.BatchNorm1d):
                m.weight.copy_(1.0 + 0.1 * torch.randn_like(m.weight))
                m.bias.copy_(0.1 * torch.randn_like(m.bias))
    sd = {k: v.detach().clone() for k, v in net.model.state_dict().items()}
    x = torch.log1p(torch.randn(B, C, T, dtype=torch.float64).abs() * 2.0)
    phi = (torch.rand(B, C, T, dtype=torch.float64) * 2 - 1) * np.pi
    with torch.backends.mkldnn.flags(enabled=False):
        out_batch = net.forward(x.clone())
        out_clip = torch.cat([net.forward(x[i:i + 1].clone()) for i in range(B)], 0)
        # train.py:45-61
        lossf = torch.nn.MSELoss()
        pp, pm = out_batch[:, :C], out_batch[:, C:]
        ang = lossf(torch.cos(pp), phi.cos()) + lossf(torch.sin(pp), phi.sin())
        mag = lossf(pm, x)
        loss = ang + mag * 0.2
        net.zero_grad()
        loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in net.model.named_parameters()}
    rec = {"x": x.numpy(), "phi": phi.numpy(), "out_batch": out_batch.detach().numpy(),
           "out_clip": out_clip.detach().numpy(), "loss": np.float64(loss.item()),
           "ang_loss": np.float64(ang.item()), "mag_loss": np.float64(mag.item()),
           "grad::model.0.weight": grads["model.0.weight"].numpy(),
           "grad::model.3.weight": grads["model.3.weight"].numpy(),
           "grad::model.1.model.3.model.3.model.3.weight":
               grads["model.1.model.3.model.3.model.3.weight"].numpy(),
           "grad::model.1.model.2.weight": grads["model.1.model.2.weight"].numpy()}
    if grad_stride > 1:
        for k in ("model.0.weight", "model.3.weight"):
            rec["grad::" + k] = rec["grad::" + k].ravel()[::grad_stride].copy()
            rec["stride::" + k] = np.int64(grad_stride)
    for k, v in sd.items():
        rec["sd::" + k] = v.numpy()
    np.savez_compressed(os.path.join(OUT, f"unet_c{C}_t{T}.npz"), **rec)
    print(f"unet_c{C}_t{T}: out {tuple(out_batch.shape)} loss {loss.item():.6f}")


def stft_case(n_fft, hop, n, seed):
    rng = np.random.default_rng(seed)
    y = (0.1 * rng.standard_normal(n) + 0.3 * np.sin(2 * np.pi * 0.01 * np.arange(n))).astype(np.float32)
    win = torch.hann_window(n_fft, periodic=True, dtype=torch.float64)
    yt = torch.from_numpy(y).double()
    S = torch.stft(yt, n_fft, hop, window=win, center=True, pad_mode="reflect", return_complex=True)
    z = torch.randn(n_fft // 2 + 1, S.shape[1], dtype=torch.complex128,
                    generator=torch.Generator().manual_seed(seed))
    z[0] = 0
    z[-1] = z[-1].real + 0j
    w = torch.istft(z, n_fft, hop, window=win, center=True, length=(S.shape[1] - 1) * hop)
    np.savez_compressed(os.path.join(OUT, f"stft_n{n_fft}_h{hop}_len{n}.npz"),
                        y=y, S=S.numpy(), z=z.numpy(), w=w.numpy())
    print(f"stft n_fft={n_fft} hop={hop} n={n}: S {tuple(S.shape)}")


def main():
    os.makedirs(OUT, exist_ok=True)
    ref_model = import_reference_model(sys.argv[1])
    unet_case(ref_model, 8, 24, 2, seed=1)
    unet_case(ref_model, 8, 40, 3, seed=2)
    unet_case(ref_model, 16, 64, 2, seed=3, grad_stride=5)
    stft_case(512, 128, 128 * 23, seed=4)
    stft_case(1024, 256, 256 * 15, seed=5)
    stft_case(2048, 512, 512 * 7, seed=6)


if __name__ == "__main__":
    main()
