"""GPU parity of the training step (train.py:37-62): loss, gradients of every parameter, Adam,
against the reference-generated golden vectors and autograd through the oracle."""
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import unet_torch  # noqa: E402

CASES = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "unet_*.npz")))


def rel_l2(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _stored_part(z, name, full):
    """The elements of ``full`` that the golden file keeps for gradient ``name``: all of them, or every
    ``stride::<name>``-th element of the flattened tensor where the file stores a strided sample (keeps it under 1 MB)."""
    key = "stride::" + name
    return full.ravel()[::int(z[key])] if key in z.files else full


def _train_py_loss(pred, x, phi, C):
    """train.py:45-60 verbatim in behaviour, with torch ops on the GPU (what a user's script does)."""
    lossf = torch.nn.MSELoss()
    pp, pm = pred[:, :C], pred[:, C:]
    ang = lossf(torch.cos(pp), phi.cos()) + lossf(torch.sin(pp), phi.sin())
    return ang + lossf(pm, x) * 0.2


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_backward_matches_reference_gradients(path):
    """loss.backward() through the drop-in model (exact-fp32 kernels at these channel counts) vs
    the gradients the real reference produced (tests/golden) and the oracle's for all parameters."""
    import model
    z = np.load(path)
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd::")}
    C = z["x"].shape[1]
    net = model.UNetModel(C, 2 * C).cuda()
    net.model.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in sd.items()})
    x = torch.from_numpy(z["x"]).float().cuda(); phi = torch.from_numpy(z["phi"]).float().cuda()
    pred = net.forward(x)
    loss = _train_py_loss(pred, x, phi, C)
    loss.backward()
    assert abs(loss.item() - float(z["loss"])) < 1e-4 * abs(float(z["loss"]))
    grads = {k: p.grad for k, p in net.model.named_parameters()}
    for k in z.files:
        if k.startswith("grad::"):
            assert rel_l2(_stored_part(z, k[6:], grads[k[6:]].cpu().numpy()), z[k]) < 2e-4, k
    tgt = torch.stack([torch.from_numpy(z["x"]), torch.from_numpy(z["phi"])], 1)
    _, _, _, ref = unet_torch.loss_and_grads(sd, torch.from_numpy(z["x"]), tgt)
    for k, g in ref.items():
        assert grads[k] is not None, k
        assert rel_l2(grads[k].cpu().numpy(), g.numpy()) < 2e-4, k


def _cos(a, b):
    a = np.asarray(a, np.float64).ravel(); b = np.asarray(b, np.float64).ravel()
    return float(np.dot(a, b) / (np.linalg.norm(a) * np.linalg.norm(b)))


@pytest.mark.parametrize("prec,tol", [("bf16x3", 1e-4), ("bf16", 2e-2)])
@pytest.mark.parametrize("T", [40, 136])
def test_tensor_core_backward_kernels_on_identical_forward_state(prec, tol, T):
    """Backward with the tensor-core kernels (wgrad_tc on MN-major operands, data gradient through
    conv_tc on the mirrored geometry) vs the exact-fp32 SIMT backward, both started from the SAME
    forward state.  (Started from their own forward passes the two differ by ~1e-2 in small layers
    because a pre-activation within the forward rounding error of zero flips a ReLU/LeakyReLU
    derivative -- a property of the network, not of the kernels; see the next test.)"""
    import model
    from phasegen import synth
    C, B = 64, 3
    torch.manual_seed(11)
    net = model.UNetModel(C, 2 * C).cuda()
    synth.randomize_norm_affine(net, seed=12)
    x = torch.log1p(torch.randn(B, C, T).abs() * 2.0).cuda()
    d_out = torch.randn(B, T, 2 * C, device="cuda") * 1e-3
    dn, up = net._norm_params(x.device)
    exs = {}
    for p in ("fp32_simt", prec):
        ex = net.train_executor(B, T, x.device, precision=p)
        ex.load_input_cf(x)
        ex.run(dn, up)
        exs[p] = ex
    ref, tc = exs["fp32_simt"], exs[prec]
    for i in range(ref.D):                      # hand the exact forward state to the tensor-core executor
        tc.z[i].copy_(ref.z[i]); tc.g[i].copy_(ref.g[i])
        for name in ("dn_ss", "dn_mv", "up_ss", "up_mv"):
            if getattr(ref, name)[i] is not None:
                getattr(tc, name)[i].copy_(getattr(ref, name)[i])
    ref.backward(dn, up, d_out=d_out); tc.backward(dn, up, d_out=d_out)
    torch.cuda.synchronize()
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    for i in range(ref.D):
        assert rel(tc.dw_up[i], ref.dw_up[i]) < tol and rel(tc.dw_dn[i], ref.dw_dn[i]) < tol, i
        assert rel(tc.din_up[i], ref.din_up[i]) < tol, i
        if ref.din_dn[i] is not None:
            assert rel(tc.din_dn[i], ref.din_dn[i]) < tol, i
        assert rel(tc.dgb_up[i][0], ref.dgb_up[i][0]) < tol and rel(tc.dgb_up[i][1], ref.dgb_up[i][1]) < tol, i


@pytest.mark.parametrize("prec,min_cos", [("bf16x3", 0.999), ("bf16", 0.98)])
def test_tensor_core_training_gradients_vs_oracle(prec, min_cos):
    """End to end (own forward pass, train.py loss, loss.backward()) against float64 autograd through
    the oracle: loss to the forward tolerance, every parameter gradient by direction (cosine), since
    isolated activation-derivative flips make an L2 bound on small tensors meaningless."""
    import model
    from phasegen import synth
    C, B, T = 64, 4, 136
    torch.manual_seed(11)
    net = model.UNetModel(C, 2 * C).cuda()
    synth.randomize_norm_affine(net, seed=12)
    net.train_precision = prec
    sd = {k: v.detach().cpu() for k, v in net.model.state_dict().items()}
    x = torch.log1p(torch.randn(B, C, T).abs() * 2.0)
    phi = (torch.rand(B, C, T) * 2 - 1) * np.pi
    pred = net.forward(x.cuda())
    loss = _train_py_loss(pred, x.cuda(), phi.cuda(), C)
    loss.backward()
    ref_loss, _, _, ref = unet_torch.loss_and_grads(sd, x, torch.stack([x, phi], 1))
    assert abs(loss.item() - ref_loss) < (1e-3 if prec == "bf16x3" else 3e-2) * abs(ref_loss)
    worst = 1.0
    for k, p in net.model.named_parameters():
        c = _cos(p.grad.cpu().numpy(), ref[k].numpy())
        worst = min(worst, c)
        assert c > min_cos, (k, c)
    print(f"{prec}: worst gradient cosine {worst:.6f}")


def test_data_gradient_of_strided_conv_with_unnatural_length():
    """The data gradient of Conv1d(k4, s2, p1) on a 29-row input (14 outputs) is a transposed
    convolution asked for one row more than its natural length (output_padding = 1)."""
    import torch.nn.functional as F
    from phasegen import ops
    B, C_in, C_out, L_in, k, s, p = 5, 128, 64, 14, 4, 2, 1       # mirrored: dZ [B,14,128] -> dX [B,29,64]
    g = torch.Generator().manual_seed(9)
    w = torch.randn(C_in, C_out, k, generator=g).cuda() / 16            # ConvTranspose1d layout [C_in][C_out][k]
    rows = 16
    x = torch.zeros(B, rows, C_in, device="cuda"); x[:, :L_in] = torch.randn(B, L_in, C_in, generator=g).cuda()
    ref = F.conv_transpose1d(x[:, :L_in].double().permute(0, 2, 1), w.double(), None, s, p, output_padding=1).permute(0, 2, 1)
    assert ref.shape[1] == 29
    # C_out 64 is not a tensor-core tile: exact SIMT kernel
    ds = ops.conv_desc(ops.PG_CONV_TRANSPOSE, B, C_in, C_out, L_in, k, s, p, rows, C_in, ops.PG_PREC_FP32_SIMT, L_out=29)
    _, _, ws = ops.pack_weight(w, ops.PG_CONV_TRANSPOSE, False, True)
    y = torch.empty(B, 29, C_out, device="cuda")
    ops.conv_simt(ds, x, ws, y)
    assert float((y.double() - ref).norm() / ref.norm()) < 2e-6
    # tensor-core kernel on a tile-sized variant
    C_out = 128
    w = torch.randn(C_in, C_out, k, generator=g).cuda() / 16
    ref = F.conv_transpose1d(x[:, :L_in].double().permute(0, 2, 1), w.double(), None, s, p, output_padding=1).permute(0, 2, 1)
    d = ops.conv_desc(ops.PG_CONV_TRANSPOSE, B, C_in, C_out, L_in, k, s, p, rows, C_in, ops.PG_PREC_BF16X3, L_out=29)
    hi, lo, _ = ops.pack_weight(w, ops.PG_CONV_TRANSPOSE)
    xh = x.to(torch.bfloat16); xl = (x - xh.float()).to(torch.bfloat16)
    y = torch.full((B, 29, C_out), float("nan"), device="cuda")
    ops.conv_tc(d, xh, xl, hi, lo, y, None)
    assert float((y.double() - ref).norm() / ref.norm()) < 3e-5


def test_loss_kernel_and_adam_kernel():
    from phasegen import ops
    B, T, C = 3, 16, 32
    g = torch.Generator().manual_seed(5)
    out = torch.randn(B, T, 2 * C, generator=g).cuda()
    lm = torch.randn(B, T, C, generator=g).abs().cuda(); ph = ((torch.rand(B, T, C, generator=g) * 2 - 1) * 3.14159).cuda()
    d_out = torch.empty_like(out); partial = torch.empty(64, 3, device="cuda", dtype=torch.float64); loss3 = torch.zeros(4, device="cuda")
    ops.phase_loss(out, lm, ph, d_out, partial, loss3)
    o = out.double().cpu().permute(0, 2, 1).requires_grad_(True)
    tgt = torch.stack([lm.double().cpu().permute(0, 2, 1), ph.double().cpu().permute(0, 2, 1)], 1)
    loss, ang, mag = unet_torch.phase_loss(o, tgt)
    loss.backward()
    assert abs(loss3[0].item() - loss.item()) < 1e-5 * loss.item()
    assert abs((loss3[1] + loss3[2]).item() - ang.item()) < 1e-5 and abs(loss3[3].item() - mag.item()) < 1e-5
    assert rel_l2(d_out.cpu().numpy(), o.grad.permute(0, 2, 1).numpy()) < 1e-5
    # Adam vs torch.optim.Adam (train.py:26-27 defaults), three steps
    p = torch.randn(1000, generator=g).cuda(); pt = p.clone().requires_grad_(True)
    m = torch.zeros_like(p); v = torch.zeros_like(p)
    opt = torch.optim.Adam([pt], lr=1e-3)
    for step in range(1, 4):
        gr = torch.randn(1000, generator=g).cuda()
        ops.adam_step(p, gr, m, v, 1e-3, 0.9, 0.999, 1e-8, step)
        pt.grad = gr.clone(); opt.step()
    assert float((p - pt.detach()).abs().max()) < 1e-6


def test_native_train_step_tracks_reference_loop():
    """TrainStep (all kernels native, Adam included) vs the reference loop restated on the CPU in
    float64: forward, train.py loss, autograd, torch.optim.Adam -- three steps on a fixed batch."""
    import model
    from phasegen.train import TrainStep
    C, B, T = 16, 2, 32
    torch.manual_seed(21)
    net = model.UNetModel(C, 2 * C).cuda()
    sd0 = {k: v.detach().cpu().clone() for k, v in net.model.state_dict().items()}
    x = torch.log1p(torch.randn(B, C, T).abs() * 2.0); phi = (torch.rand(B, C, T) * 2 - 1) * np.pi
    step = TrainStep(net, B, T, "cuda", precision="fp32_simt", lr=1e-3)
    lm_cl = x.permute(0, 2, 1).contiguous().cuda(); ph_cl = phi.permute(0, 2, 1).contiguous().cuda()
    losses = [float(step(lm_cl, ph_cl)[0]) for _ in range(3)]
    # reference loop
    keys = [k for k, v in sd0.items() if v.is_floating_point() and "running_" not in k]
    leaf = {k: sd0[k].double().clone().requires_grad_(True) for k in keys}
    opt = torch.optim.Adam(list(leaf.values()), lr=1e-3)
    ref_losses = []
    for _ in range(3):
        opt.zero_grad()
        full = dict(sd0); full.update(leaf)
        with torch.backends.mkldnn.flags(enabled=False):
            out = unet_torch.unet_forward(full, x, torch.float64, grad=True)
            loss, _, _ = unet_torch.phase_loss(out, torch.stack([x, phi], 1).double())
            loss.backward()
        opt.step()
        ref_losses.append(loss.item())
    assert np.allclose(losses, ref_losses, rtol=2e-4), (losses, ref_losses)
    assert ref_losses[2] < ref_losses[0]
    w = net.model.state_dict()["model.3.weight"].cpu().double()
    assert rel_l2(w.numpy(), leaf["model.3.weight"].detach().numpy()) < 1e-4


def test_optimizer_state_round_trip_resumes_identically(tmp_path):
    """TrainStep.state_dict()/load_state_dict(): a run resumed from (model checkpoint, optimiser state) continues
    bit-identically to the uninterrupted one, and the state file is in the torch layout of each parameter."""
    import model
    from phasegen.train import TrainStep
    C, T, B = 64, 32, 4
    torch.manual_seed(21)
    lm = torch.rand(B, T, C, device="cuda") * 3
    ph = (torch.rand(B, T, C, device="cuda") - 0.5) * 6
    net = model.UNetModel(C, 2 * C).cuda()
    step = TrainStep(net, B, T, "cuda", precision="bf16x3")
    for _ in range(3):
        step(lm, ph)
    ck = str(tmp_path / "ckpt")
    net.save(ck)
    opt = step.state_dict()
    torch.save(opt, str(tmp_path / "opt"))
    assert opt["step"] == 3
    w = dict(net.model.named_parameters())
    for name, st in opt["state"].items():
        assert tuple(st["exp_avg"].shape) == tuple(w[name].shape), name
    a = [float(step(lm, ph)[0]) for _ in range(3)]
    net2 = model.UNetModel(C, 2 * C).cuda()
    net2.load(ck)
    step2 = TrainStep(net2, B, T, "cuda", precision="bf16x3")
    step2.load_state_dict(torch.load(str(tmp_path / "opt")))
    b = [float(step2(lm, ph)[0]) for _ in range(3)]
    assert a == b


def test_bf16_gradient_path_tracks_the_fp32_one():
    """grad_dtype="bf16" (the data-parallel default: wgrad writes bf16, NCCL would reduce bf16, Adam reads bf16)
    against fp32 gradients from the same start: same loss trajectory to bf16 rounding of the gradients."""
    import copy
    import model
    from phasegen.train import TrainStep
    C, T, B = 128, 32, 4
    torch.manual_seed(23)
    lm = torch.rand(B, T, C, device="cuda") * 3
    ph = (torch.rand(B, T, C, device="cuda") - 0.5) * 6
    net_a = model.UNetModel(C, 2 * C).cuda()
    net_b = model.UNetModel(C, 2 * C).cuda()
    net_b.model.load_state_dict(copy.deepcopy(net_a.model.state_dict()))
    sa = TrainStep(net_a, B, T, "cuda", precision="bf16x3", grad_dtype="fp32")
    sb = TrainStep(net_b, B, T, "cuda", precision="bf16x3", grad_dtype="bf16")
    assert sb.ex.dw_up[0].dtype == torch.bfloat16 and sa.ex.dw_up[0].dtype == torch.float32
    la = [float(sa(lm, ph)[0]) for _ in range(6)]
    lb = [float(sb(lm, ph)[0]) for _ in range(6)]
    assert la[0] == lb[0]                                        # identical forward before the first update
    assert la[-1] < la[0] and lb[-1] < lb[0]
    assert max(abs(a - b) / a for a, b in zip(la, lb)) < 2e-3
    wa = net_a.model.model[0].weight.detach().float(); wb = net_b.model.model[0].weight.detach().float()
    assert float((wa - wb).norm() / wa.norm()) < 2e-3


def test_async_checkpoint_equals_sync_checkpoint(tmp_path):
    """UNetModel.save_async: same file content as save(), written while the GPU keeps working."""
    import model
    net = model.UNetModel(64, 128).cuda()
    x = torch.randn(2, 64, 32, device="cuda")
    net.forward(x)                                              # moves the running statistics
    h = net.save_async(str(tmp_path / "a"))
    net.forward(x)                                              # work queued behind the snapshot must not leak into it
    net.save(str(tmp_path / "b_after"))
    h.wait()
    a = torch.load(str(tmp_path / "a"))
    net2 = model.UNetModel(64, 128).cuda()
    net2.load(str(tmp_path / "a"))
    for k, v in net2.model.state_dict().items():
        assert torch.equal(v.cpu(), a[k]), k
    b = torch.load(str(tmp_path / "b_after"))
    assert set(a) == set(b)
    assert int(a["model.4.num_batches_tracked"]) + 1 == int(b["model.4.num_batches_tracked"])
    assert torch.equal(a["model.0.weight"], b["model.0.weight"])


def test_config3_shape_training_parity():
    """BASELINE.json config 3 at its own shape -- UNetModel(1024, 2048), 128-frame pairs, bf16 products and bf16 weight
    gradients (batch 8 instead of 32 to keep the checker quick; tile plans depend on B only through the tile count).
    This shape takes code paths the small cases do not: merged-clip MMAs with two MMA groups per weight tile, 512-column
    accumulators, the wide (256 input channels x 2 taps) weight-gradient form, CTA pairs in forward and data gradient.
      (a) forward vs the float64 oracle (run on the GPU in float64: same restatement, torch does the arithmetic);
          bound 3e-2 relative L2 on the network output = the separately stated loose bf16 bound;
      (b) every data / weight gradient of the tensor-core kernels vs the exact-fp32 SIMT kernels from an IDENTICAL
          forward state, bound 2e-2 (bf16 operand rounding, bf16 gradient storage);
      (c) one TrainStep vs a float64 reference step: loss within 3e-2, every weight gradient by direction
          (cosine >= 0.98), the first Adam update (-lr * g / (|g| + eps)) by direction (cosine >= 0.85, measured 0.90 on the smallest-gradient layer: elements whose
          gradient is within the bf16 noise of zero flip the sign of their +-lr update)."""
    import model
    from phasegen import synth
    from phasegen.train import TrainStep
    C, T, B = 1024, 128, 8
    dev = torch.device("cuda")
    torch.manual_seed(21)
    net = model.UNetModel(C, 2 * C).to(dev)
    synth.randomize_norm_affine(net, seed=22)
    sd = {k: v.detach().clone() for k, v in net.model.state_dict().items()}
    g = torch.Generator().manual_seed(23)
    sigma = 4.0 / (1.0 + torch.arange(C, dtype=torch.float32) / 32.0)
    re, im = torch.randn(B, T, C, generator=g) * sigma, torch.randn(B, T, C, generator=g) * sigma
    lm = torch.log1p(torch.sqrt(re * re + im * im)).contiguous().to(dev)
    ph = torch.atan2(im, re).contiguous().to(dev)
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    cos = lambda a, b: float(torch.dot(a.double().reshape(-1), b.double().reshape(-1)) / (a.double().norm() * b.double().norm()))

    # ---- float64 reference (oracle on the GPU): forward, loss, gradients
    x_cf = lm.permute(0, 2, 1).contiguous().double()
    target = torch.stack([x_cf, ph.permute(0, 2, 1).double()], 1)
    ref_out = unet_torch.unet_forward(sd, x_cf, torch.float64)
    ref_loss, _, _, ref_g = unet_torch.loss_and_grads(sd, x_cf, target, torch.float64)

    # ---- (a) forward
    dn, up = net._norm_params(dev)
    tc = net.train_executor(B, T, dev, precision="bf16", grad_dtype=torch.bfloat16)
    tc.load_input_cl(lm)
    tc.run(dn, up)
    e_out = rel(tc.out.permute(0, 2, 1), ref_out)
    print(f"config-3 shape forward (bf16) vs float64 oracle: rel-L2 {e_out:.2e}")
    assert e_out < 3e-2

    # ---- (b) backward kernels on an identical forward state
    simt = net.train_executor(B, T, dev, precision="fp32_simt")
    simt.load_input_cl(lm)
    simt.run(dn, up)
    for i in range(simt.D):
        tc.z[i].copy_(simt.z[i]); tc.g[i].copy_(simt.g[i])
        for name in ("dn_ss", "dn_mv", "up_ss", "up_mv"):
            if getattr(simt, name)[i] is not None:
                getattr(tc, name)[i].copy_(getattr(simt, name)[i])
    d_out = torch.randn(B, T, 2 * C, device=dev, generator=torch.Generator(device=dev).manual_seed(24)) * 1e-3
    simt.backward(dn, up, d_out=d_out); tc.backward(dn, up, d_out=d_out)
    torch.cuda.synchronize()
    worst = 0.0
    for i in range(simt.D):
        errs = [rel(tc.dw_up[i], simt.dw_up[i]), rel(tc.dw_dn[i], simt.dw_dn[i]), rel(tc.din_up[i], simt.din_up[i])]
        if simt.din_dn[i] is not None:
            errs.append(rel(tc.din_dn[i], simt.din_dn[i]))
        worst = max(worst, max(errs))
        assert max(errs) < 2e-2, (i, errs)
    print(f"config-3 shape wgrad/dgrad (bf16, bf16 gradients) vs exact SIMT: worst rel-L2 {worst:.2e}")
    del simt
    net.__dict__["_exec"] = {k: v for k, v in net._exec.items() if v is tc}

    # ---- (c) one optimisation step
    w_before = {k: p.detach().clone() for k, p in net.model.named_parameters()}
    step = TrainStep(net, B, T, dev, precision="bf16")
    assert step.ex is tc and step.grad_dtype == torch.bfloat16
    loss3 = step(lm, ph)
    torch.cuda.synchronize()
    assert abs(float(loss3[0]) - ref_loss) < 3e-2 * abs(ref_loss), (float(loss3[0]), ref_loss)
    grads = dict(zip((n for n, _ in net.model.named_parameters()), net._param_grads(tc)))
    lr, eps = 1e-3, 1e-8
    worst_g, worst_u = 1.0, 1.0
    for k, p in net.model.named_parameters():
        assert bool(torch.isfinite(p).all()), k
        rg = ref_g[k]
        c_g = cos(grads[k].float(), rg)
        d_ref = -lr * rg / (rg.abs() + eps)
        c_u = cos(p.detach() - w_before[k], d_ref)
        worst_g, worst_u = min(worst_g, c_g), min(worst_u, c_u)
        assert c_g > 0.98, (k, c_g)
        assert c_u > 0.85, (k, c_u)
    print(f"config-3 shape TrainStep vs float64 step: loss {float(loss3[0]):.5f} vs {ref_loss:.5f}, worst gradient cosine "
          f"{worst_g:.4f}, worst update cosine {worst_u:.4f}")


def test_backward_after_a_second_forward_raises():
    """One set of activation buffers per shape: a backward whose forward state was overwritten by a later forward of the
    same shape must raise instead of returning gradients of the wrong graph; forward/backward pairs accumulate fine."""
    import model
    C, B, T = 8, 2, 24
    torch.manual_seed(3)
    net = model.UNetModel(C, 2 * C).cuda()
    x1, x2 = torch.randn(B, C, T, device="cuda"), torch.randn(B, C, T, device="cuda")
    y1 = net.forward(x1)
    y2 = net.forward(x2)
    with pytest.raises(RuntimeError, match="overwritten by a later forward"):
        (y1.sum() + y2.sum()).backward()
    net.zero_grad()
    net.forward(x1).sum().backward()
    g1 = [p.grad.clone() for p in net.parameters()]
    net.forward(x2).sum().backward()                       # accumulates into p.grad like any autograd node
    net.zero_grad()
    net.forward(x2).sum().backward()
    g2 = [p.grad.clone() for p in net.parameters()]
    net.zero_grad()
    net.forward(x1).sum().backward(); net.forward(x2).sum().backward()
    for p, a, b in zip(net.parameters(), g1, g2):
        assert torch.allclose(p.grad, a + b, rtol=1e-5, atol=1e-6)


def test_async_checkpoint_is_a_snapshot_of_the_call_time(tmp_path):
    """save_async on a model large enough (C = 512: 0.6 GB) that the pinned-host copy is still in flight when the
    weights are overwritten right after the call: the file must hold the weights of the call time, not a mixture."""
    import model
    torch.manual_seed(5)
    net = model.UNetModel(512, 1024).cuda()
    want = {k: v.detach().cpu().clone() for k, v in net.model.state_dict().items()}
    path = str(tmp_path / "snap.pt")
    h = net.save_async(path)
    with torch.no_grad():
        for p in net.parameters():
            p.add_(1.0)                                    # the "next optimiser step", queued immediately
    h.wait()
    got = torch.load(path, map_location="cpu")
    assert set(got) == set(want)
    for k in want:
        assert torch.equal(got[k], want[k]), k


def test_host_batch_feeder_prefetches_in_order():
    """HostBatchFeeder: batches prefetched from pinned host memory come back in order, each in its own device slot, with
    the slot of a batch reused only after `done()`; a third prefetch without a `next()` is refused."""
    from phasegen.train import HostBatchFeeder
    shape = (3, 16, 64)
    feeder = HostBatchFeeder(shape, "cuda")
    hosts = [(torch.full(shape, float(i)).pin_memory(), torch.full(shape, float(-i)).pin_memory()) for i in range(5)]
    feeder.prefetch(*hosts[0])
    seen = []
    for i in range(5):
        lm, ph = feeder.next()
        seen.append((float(lm.sum()), float(ph.sum())))          # consumed on the current stream, after the copy
        feeder.done()
        if i + 1 < 5:
            feeder.prefetch(*hosts[i + 1])
    n = 3 * 16 * 64
    assert seen == [(float(i * n), float(-i * n)) for i in range(5)]
    feeder.prefetch(*hosts[0]); feeder.prefetch(*hosts[1])
    with pytest.raises(RuntimeError, match="not been consumed"):
        feeder.prefetch(*hosts[2])
    a, _ = feeder.next()
    assert float(a.sum()) == 0.0
