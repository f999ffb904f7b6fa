"""GPU: the pixel decoder (csrc/deconv.cu) layer by layer through the C ABI (`rlrep_conv_decoder_*`) against plain
float64 PyTorch restatements of the reference modules: muLV-Rep's Decoder (agent/mulvdrq/drqv2.py:98-117, as
oracle/mulv_oracle.py:78-82 writes it; output kernel 2, L1 loss of :180) and the latent Diff-SR VAE decoder's
convolutions (vae_1d.Decoder, oracle/ldiffsr_oracle.py:104-110; output kernel 3, summed MSE loss of :204).

Per-layer checks feed each float64 reference layer with the kernel's OWN input map (act_l, or dact_{l+1} and act_l
backwards), so every comparison holds exactly one layer of rounding and there is no ReLU flip to excuse: the ReLU mask
the reference applies is `act_l > 0` of the very map the kernel masked with.  Errors are rel-L2 over the whole map and,
separately, over every frame, over the 2-pixel border band and over each (y % 2, x % 2) class of the 83/84-wide maps
(the stride-2 layer's parity classes): an error confined to one row, column, frame or class cannot hide in a norm.

Bars, about 3x the worst value measured on one NVIDIA B200 (1000 W power limit) over every case below:
- per layer and per slice: fp32 1e-5 (worst 3.3e-6: the output layer's bias gradient, a sum over 48 x 84 x 84 pixels;
  maps and weight gradients stay below 2.3e-6), tf32 1.2e-3 (worst 4.1e-4: a parity class of the stride-2 output;
  weight gradients stay below 3.0e-4, at 1024 frames);
- loss values 2e-6 (worst 6.7e-7) and loss gradients 2e-7 (worst 6.7e-8): fp32 CUDA-core kernels at either precision;
- end to end, test_decoder_end_to_end.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

IN_DIM = 32 * 35 * 35
PAD = 36  # row pitch IN_DIM + PAD, as the agents pass their F_-wide buffers
DX_SENTINEL = 1234.5
BAR = {"fp32": 1e-5, "tf32": 1.2e-3}
LOSS_BAR, DPRED_BAR = 2e-6, 2e-7  # the loss kernels run in fp32 on CUDA cores whatever the handle's precision
CHUNK = 256  # frames per float64 reference pass


# ------------------------------------------------------------------------------------------------ references
def ref_layer(l, x, sd, ks, relu=True):
    """Layer l of the decoder on a float64 NCHW map: ConvTranspose2d (+ ReLU) for l = 0..3, the output Conv2d for l = 4."""
    w, b = sd[f"deconvnet.{2 * l}.weight"], sd[f"deconvnet.{2 * l}.bias"]
    if l == 4:
        return F.conv2d(x, w, b, padding=1)
    y = F.conv_transpose2d(x, w, b, stride=2 if l == 3 else 1, output_padding=1 if (l == 3 and ks == 3) else 0)
    return F.relu(y) if relu else y


def ref_decoder(sd, x, ks):
    h = x.view(x.shape[0], 32, 35, 35)
    for l in range(4):
        h = ref_layer(l, h, sd, ks)
    return ref_layer(4, h, sd, ks)


def l1_target(t):
    return t.float() / 255.0 - 0.5  # fp32, as the oracle computes it from the uint8 frame (mulv_oracle.py:180)


def mse_target(t, shifts):
    """The shift-augmented frame (RandomShiftsAug with integer shifts == replicate padding and a crop) / 255 - 0.5 in
    fp32 (ldiffsr_oracle.py:196, 204); shifts [B, 2] = (x, y) in [0, 8]."""
    f = t.float()
    if shifts is not None:
        p = F.pad(f, (4, 4, 4, 4), mode="replicate")
        f = torch.stack([p[b, :, sy:sy + 84, sx:sx + 84] for b, (sx, sy) in enumerate(shifts.tolist())])
    return f / 255.0 - 0.5


def ref_loss(kind, pred, target, shifts, grad_scale):
    """(loss, grad_scale * d loss / d pred) in float64 from a given prediction (mulv_oracle.py:180, ldiffsr_oracle.py:204)."""
    B = pred.shape[0]
    if kind == "l1":
        d = pred.double() - l1_target(target).double()
        return 10.0 * d.abs().mean().item(), torch.sign(d) * (grad_scale * 10.0 / d.numel())
    d = pred.double() - mse_target(target, shifts).double()
    return (d * d).sum().item() / B, d * (2.0 * grad_scale / B)


# ------------------------------------------------------------------------------------------------ error measures
def rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def slice_errors(out, ref):
    """rel-L2 over the whole map and the worst over frames, the 2-pixel border band and, on the 83/84-wide maps, the four
    (y % 2, x % 2) classes."""
    e = (out.double() - ref.double()) ** 2
    r = ref.double() ** 2

    def q(num, den):
        return math.sqrt(num) / max(math.sqrt(den), 1e-300) if num > 0 else 0.0
    errs = {"all": q(e.sum().item(), r.sum().item())}
    num_f, den_f = e.sum(dim=(1, 2, 3)), r.sum(dim=(1, 2, 3))
    errs["frame"] = max(q(n, d) for n, d in zip(num_f.tolist(), den_f.tolist()))
    H, W = out.shape[-2:]
    band = torch.ones(H, W, dtype=torch.bool, device=out.device)
    band[2:H - 2, 2:W - 2] = False
    errs["border"] = q(e[..., band].sum().item(), r[..., band].sum().item())
    if H >= 83:
        errs["parity"] = max(q(e[..., py::2, px::2].sum().item(), r[..., py::2, px::2].sum().item())
                             for py in (0, 1) for px in (0, 1))
    return errs


# ------------------------------------------------------------------------------------------------ fixtures
def make_params(ks, regime, seed):
    """He-scaled signed weights ("realistic"), or non-negative ones behind a +8 bias ("all_active": every pre-activation
    of the four transposed layers is positive, so no ReLU mask is ever zero)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for l in range(4):
        w = torch.randn(32, 32, 3, 3, generator=g) * (2.0 / 288) ** 0.5
        b = torch.randn(32, generator=g) * 0.1
        if regime == "all_active":
            w, b = w.abs() / 8, b + 8.0
        sd[f"deconvnet.{2 * l}.weight"], sd[f"deconvnet.{2 * l}.bias"] = w, b
    sd["deconvnet.8.weight"] = torch.randn(3, 32, ks, ks, generator=g) * (2.0 / (32 * ks * ks)) ** 0.5
    sd["deconvnet.8.bias"] = torch.randn(3, generator=g) * 0.1
    return sd


def make_inputs(B, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, IN_DIM, generator=g)
    target = torch.randint(0, 256, (B, 3, 84, 84), generator=g, dtype=torch.uint8)
    shifts = torch.randint(0, 9, (B, 2), generator=g, dtype=torch.int32)
    extremes = torch.tensor([[0, 0], [8, 8], [0, 8], [8, 0]], dtype=torch.int32)
    shifts[:min(B, 4)] = extremes[:min(B, 4)]
    return x, target, shifts


def pitched(x, fill):
    """x [B, IN_DIM] as a view of rows IN_DIM + PAD wide whose padding columns hold `fill`."""
    full = torch.full((x.shape[0], IN_DIM + PAD), fill, device="cuda")
    full[:, :IN_DIM] = x.cuda()
    return full, full[:, :IN_DIM]


def run_decoder(dec, sd, x, target, shifts, loss, grad_scale):
    """forward -> loss -> backward on pitched buffers; returns (loss value, dx_full)."""
    dec.load_state_dict(sd)
    _, xv = pitched(x, float("nan"))
    dec.forward(xv)
    if loss == "l1":
        lv = dec.l1_loss(target.cuda(), grad_scale)
    else:
        lv = dec.mse_sum_loss(target.cuda(), shifts.cuda() if shifts is not None else None, grad_scale)
    dx_full, dxv = pitched(torch.zeros(x.shape[0], IN_DIM), DX_SENTINEL)
    dec.backward(dxv)
    torch.cuda.synchronize()
    return lv, dx_full


def chunks(B):
    return [(i, min(i + CHUNK, B)) for i in range(0, B, CHUNK)]


def per_layer_errors(dec, sd, ks, B, loss, target, shifts, grad_scale, dx_full):
    """Every comparison of the module docstring, on a handle that has run forward, loss and backward."""
    sd64 = {k: v.double().cuda() for k, v in sd.items()}
    grads = dec.grads()
    errs = {}
    acts = [dec.read_map("act", i) for i in range(5)]
    dacts = [dec.read_map("dact", i) for i in range(5)]
    pred, dpred = dec.read_map("pred"), dec.read_map("dpred")
    outs = acts[1:] + [pred]
    for l in range(5):
        # forward: the reference layer fed with the kernel's own input
        ref = torch.cat([ref_layer(l, acts[l][a:b].double(), sd64, ks) for a, b in chunks(B)])
        errs[f"fwd{l}"] = slice_errors(outs[l], ref)
        del ref
        # backward: from the kernel's own dact_{l+1} (dpred for the output layer) and act_l
        gy = dacts[l + 1] if l < 4 else dpred
        W = sd64[f"deconvnet.{2 * l}.weight"].clone().requires_grad_()
        bb = sd64[f"deconvnet.{2 * l}.bias"].clone().requires_grad_()
        dx_ref = []
        for a, b in chunks(B):
            xin = acts[l][a:b].double().requires_grad_()
            y = ref_layer(l, xin, {f"deconvnet.{2 * l}.weight": W, f"deconvnet.{2 * l}.bias": bb}, ks, relu=False)
            y.backward(gy[a:b].double())
            dx_ref.append(xin.grad * (acts[l][a:b] > 0) if l > 0 else xin.grad)
        dx_ref = torch.cat(dx_ref)
        errs[f"dact{l}"] = slice_errors(dacts[l], dx_ref)
        errs[f"dW{l}"] = {"all": rel(grads[f"deconvnet.{2 * l}.weight"].cuda(), W.grad)}
        errs[f"db{l}"] = {"all": rel(grads[f"deconvnet.{2 * l}.bias"].cuda(), bb.grad)}
        if l == 0:
            errs["dx"] = slice_errors(dx_full[:, :IN_DIM].reshape(B, 32, 35, 35), dx_ref)
        del dx_ref
    # the loss kernel from the kernel's own prediction
    lv_ref, dpred_ref = ref_loss(loss, pred, target.cuda(), shifts.cuda() if shifts is not None else None, grad_scale)
    return errs, acts, pred, dpred, dpred_ref, lv_ref


def worst(errs):
    return max(v for e in errs.values() for v in e.values())


def fmt(errs):
    return ", ".join(f"{k} " + "/".join(f"{v:.1e}" for v in e.values()) for k, e in errs.items())


# ------------------------------------------------------------------------------------------------ per-layer tests
CASES = [(ks, prec, B, "realistic") for ks in (2, 3) for prec in ("fp32", "tf32") for B in (1, 3, 4, 6, 48, 64, 256)]
CASES += [(ks, prec, B, "all_active") for ks in (2, 3) for prec in ("fp32", "tf32") for B in (4, 48)]
CASES += [(3, "tf32", 1024, "realistic")]  # Latent Diff-SR's bench decodes 4 x 256 frames


@pytest.mark.parametrize("ks,precision,batch,regime", CASES)
def test_decoder_layers_match_float64(ks, precision, batch, regime):
    """Per-layer forward and backward, the loss kernel of the agent that uses this output kernel (L1 for 2, summed MSE
    with shifts for 3), and dx at the caller's row pitch.  The decoder input's padding columns hold NaN (they must not
    reach any output) and dx's padding columns a sentinel (they must be left as they are)."""
    from rlrep_b200.pixel import ConvDecoder
    loss = "l1" if ks == 2 else "mse"
    grad_scale = 0.5 if loss == "l1" else 0.75
    sd = make_params(ks, regime, seed=ks * 1000 + batch)
    x, target, shifts = make_inputs(batch, seed=ks * 1000 + batch + 1)
    dec = ConvDecoder(batch=batch, out_kernel=ks, precision=precision)
    lv, dx_full = run_decoder(dec, sd, x, target, shifts, loss, grad_scale)
    for k, v in dec.state_dict().items():
        assert torch.equal(v, sd[k]), k  # layout round trip through the C ABI
    errs, acts, pred, dpred, dpred_ref, lv_ref = per_layer_errors(dec, sd, ks, batch, loss, target, shifts, grad_scale,
                                                                  dx_full)
    assert torch.equal(acts[0], x.cuda().view(batch, 32, 35, 35))  # the pitched input, NCHW -> NHWC
    loss_err = abs(lv - lv_ref) / abs(lv_ref)
    if loss == "l1":  # the signs exactly, the common magnitude to fp32 rounding
        assert torch.equal(torch.sign(dpred.double()), torch.sign(dpred_ref))
        dpred_err = rel(dpred.abs(), dpred_ref.abs())
    else:
        dpred_err = rel(dpred, dpred_ref)
    print(f"\nKS={ks} {precision} B={batch} {regime}: loss {loss_err:.1e} dpred {dpred_err:.1e} | {fmt(errs)}")
    print(f"WORST ks={ks} {precision} B={batch} {regime} {worst(errs):.3e}")
    # the NaN padding of x reaches nothing, dx's padding columns are untouched
    for t in acts + [pred, dpred, dx_full[:, :IN_DIM]]:
        assert torch.isfinite(t).all()
    assert torch.all(dx_full[:, IN_DIM:] == DX_SENTINEL)
    for g in dec.grads().values():
        assert torch.isfinite(g).all()
    assert loss_err < LOSS_BAR and dpred_err < DPRED_BAR, (loss_err, dpred_err)
    bad = {k: e for k, e in errs.items() if max(e.values()) >= BAR[precision]}
    assert not bad, bad
    dec.close()


@pytest.mark.parametrize("ks", [2, 3])
def test_decoder_loss_kernels(ks):
    """Both loss kernels on one handle, from its own prediction: L1 (exact signs), MSE without shifts and MSE with shifts
    that include the extremes 0 and 8 on both axes (the clamped lookup of replicate padding)."""
    from rlrep_b200.pixel import ConvDecoder
    B = 8
    sd = make_params(ks, "realistic", seed=77 + ks)
    x, target, shifts = make_inputs(B, seed=78 + ks)
    shifts[4:8] = torch.tensor([[0, 3], [8, 5], [2, 0], [6, 8]], dtype=torch.int32)
    dec = ConvDecoder(batch=B, out_kernel=ks, precision="fp32")
    dec.load_state_dict(sd)
    dec.forward(x.cuda())
    pred = dec.read_map("pred")
    for kind, sh, gs in (("l1", None, 0.5), ("mse", None, 1.0), ("mse", shifts, 0.75)):
        lv = dec.l1_loss(target.cuda(), gs) if kind == "l1" else dec.mse_sum_loss(
            target.cuda(), sh.cuda() if sh is not None else None, gs)
        dpred = dec.read_map("dpred")
        lv_ref, dpred_ref = ref_loss(kind, pred, target.cuda(), sh.cuda() if sh is not None else None, gs)
        loss_err = abs(lv - lv_ref) / abs(lv_ref)
        if kind == "l1":
            assert torch.equal(torch.sign(dpred.double()), torch.sign(dpred_ref))
            dpred_err = rel(dpred.abs(), dpred_ref.abs())
        else:
            dpred_err = rel(dpred, dpred_ref)
            if sh is not None:  # a shifted target must differ from the unshifted one where the check could tell
                assert rel(dpred_ref, ref_loss(kind, pred, target.cuda(), None, gs)[1]) > 1e-2
        print(f"\nKS={ks} {kind} shifts={sh is not None}: loss {loss_err:.1e} dpred {dpred_err:.1e}")
        assert loss_err < LOSS_BAR and dpred_err < DPRED_BAR, (kind, loss_err, dpred_err)
    dec.close()


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("ks,batch", [(2, 6), (2, 64), (3, 6), (3, 64)])
@pytest.mark.parametrize("regime", ["all_active", "realistic"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_decoder_end_to_end(ks, batch, regime, precision):
    """x -> pred -> loss -> dx and all ten parameter gradients against one float64 autograd pass.
    all_active: every ReLU mask is all ones and |pred| >> |target| (so no L1 sign is in doubt): the agent's own loss
      (L1 for output kernel 2, MSE for 3), everything held to the precision's bar.
    realistic: He-scaled signed weights, half the units masked, summed MSE for both output kernels.  The forward pass
      keeps the bar.  The gradient of a ReLU network is discontinuous: a pre-activation within rounding distance of
      zero flips its mask between two correct implementations, and each flip moves the gradient by a whole upstream
      entry (under TF32 operand rounding about 1e-3 of the units sit that close) -- the same argument as the encoder's
      test (test_gpu_conv.py) -- so gradients are held to 5e-3 (fp32) / 6e-2 (tf32).  L1 is left out of this regime
      because a sign flip of pred - target is the same kind of discontinuity one layer later; the per-layer test checks
      the L1 kernel exactly from the kernel's own prediction.
    Measured on one NVIDIA B200 (1000 W power limit), worst over these cases: prediction 6.1e-7 (fp32) / 7.8e-4 (tf32,
    five layers of operand rounding); all_active gradients 2.7e-6 / 3.5e-4; realistic gradients 1.3e-3 / 2.6e-2 (dx,
    where the mask flips of all four ReLU layers meet).  Bars: prediction and loss 2e-6 / 2e-3, all_active gradients
    1e-5 / 1e-3, realistic gradients 5e-3 / 6e-2."""
    from rlrep_b200.pixel import ConvDecoder
    loss = "l1" if (ks == 2 and regime == "all_active") else "mse"
    grad_scale = 0.5
    sd = make_params(ks, regime, seed=500 + ks * 10 + batch)
    x, target, shifts = make_inputs(batch, seed=501 + ks * 10 + batch)
    if loss == "l1":
        shifts = None
    dec = ConvDecoder(batch=batch, out_kernel=ks, precision=precision)
    lv, dx_full = run_decoder(dec, sd, x, target, shifts, loss, grad_scale)
    pred, grads = dec.read_map("pred"), dec.grads()

    p = {k: v.double().cuda().requires_grad_() for k, v in sd.items()}
    xr = x.double().cuda().requires_grad_()
    pred_ref = ref_decoder(p, xr, ks)
    if loss == "l1":
        lref = 10.0 * (pred_ref - l1_target(target.cuda()).double()).abs().mean()
    else:
        lref = ((pred_ref - mse_target(target.cuda(), shifts.cuda()).double()) ** 2).sum() / batch
    (lref * grad_scale).backward()
    errs = {"pred": rel(pred, pred_ref.detach()), "loss": abs(lv - lref.item()) / abs(lref.item()),
            "dx": rel(dx_full[:, :IN_DIM], xr.grad)}
    for k in sd:
        errs[k] = rel(grads[k].cuda(), p[k].grad)
    print(f"\nKS={ks} B={batch} {regime} {precision}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    fp32 = precision == "fp32"
    assert errs["pred"] < (2e-6 if fp32 else 2e-3) and errs["loss"] < (2e-6 if fp32 else 2e-3), errs
    if regime == "all_active":
        grad_bar = 1e-5 if fp32 else 1e-3
    else:
        grad_bar = 5e-3 if fp32 else 6e-2
    assert max(v for k, v in errs.items() if k not in ("pred", "loss")) < grad_bar, errs
    dec.close()


# ------------------------------------------------------------------------------------------------ state
@pytest.mark.parametrize("ks,precision,batch", [(2, "tf32", 48), (3, "fp32", 6), (3, "tf32", 64)])
def test_decoder_deterministic_and_stateless(ks, precision, batch):
    """Two identical forward + loss + backward calls give bit-identical results, and a handle that first ran other
    weights and inputs gives results bit-identical to a fresh handle."""
    from rlrep_b200.pixel import ConvDecoder
    loss = "l1" if ks == 2 else "mse"
    sd = make_params(ks, "realistic", seed=900 + batch)
    x, target, shifts = make_inputs(batch, seed=901 + batch)
    sd_o = make_params(ks, "all_active", seed=902 + batch)
    x_o, target_o, shifts_o = make_inputs(batch, seed=903 + batch)

    def outputs(dec):
        lv, dx_full = run_decoder(dec, sd, x, target, shifts, loss, 0.5)
        maps = [dec.read_map(w, i) for w in ("act", "dact") for i in range(5)] + [dec.read_map("pred"),
                                                                                  dec.read_map("dpred")]
        return [torch.tensor([lv]), dx_full.cpu()] + [m.cpu() for m in maps] + list(dec.grads().values())

    used = ConvDecoder(batch=batch, out_kernel=ks, precision=precision)
    run_decoder(used, sd_o, x_o * 3.0, target_o, shifts_o, loss, 2.0)
    a, b = outputs(used), outputs(used)
    fresh = ConvDecoder(batch=batch, out_kernel=ks, precision=precision)
    c = outputs(fresh)
    for i, (u, v, w) in enumerate(zip(a, b, c)):
        assert torch.equal(u, v), f"output {i} differs between two identical calls"
        assert torch.equal(u, w), f"output {i} differs between a used and a fresh handle"
    used.close()
    fresh.close()


# ------------------------------------------------------------------------------------------------ coverage
def test_decoder_paths_are_reached():
    """The shapes of this file reach every decoder path: the halo kernel (stride-2 and stride-1 layers from B ~ 38-56 on),
    the SIMT convolutions and compaction below that and in fp32, the column-matrix stride-2 forward, the strided im2col
    with folded (rows % 4 == 0) and plain weight gradients, the implicit weight gradient, and both output kernels.  If
    the planner stops reaching one of them at these sizes, this test says so."""
    from torch.profiler import ProfilerActivity, profile
    from rlrep_b200.pixel import ConvDecoder
    names = set()
    for ks in (2, 3):
        for precision in ("fp32", "tf32"):
            for batch in (4, 6, 48, 64):
                loss = "l1" if ks == 2 else "mse"
                sd = make_params(ks, "realistic", seed=ks + batch)
                x, target, shifts = make_inputs(batch, seed=ks + batch + 1)
                dec = ConvDecoder(batch=batch, out_kernel=ks, precision=precision)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    run_decoder(dec, sd, x, target, shifts, loss, 0.5)
                    torch.cuda.synchronize()
                names |= {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
                dec.close()
    want = ["gemm_conv_halo", "compact_grid", "col2im_bias_relu", "im2col_strided", "diag_block_sum", "diag_tap_sum"]
    want += [f"out_conv_{p}_kernel<{k}>" for p in ("fwd", "dgrad", "wgrad", "wgrad_finish") for k in (2, 3)]
    missing = [w for w in want if not any(w in n for n in names)]
    simt = [n for n in names if any(s in n for s in ("gemm_tiled_kernel", "skinny_rowwarp_kernel", "skinny_rowthread_kernel"))]
    print("\n" + "\n".join(sorted(n[:160] for n in names)))
    assert not missing, missing
    assert simt, "no SIMT GEMM kernel ran"
