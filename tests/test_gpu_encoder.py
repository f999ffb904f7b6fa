"""GPU: the pixel encoder (csrc/conv.cu, csrc/conv_implicit.cu) layer by layer through the C ABI
(`rlrep_conv_encoder_*`) against plain float64 PyTorch restatements of the reference's Encoder
(network_arch/drqv2.py:138-167; RandomShiftsAug with integer shifts, :21-57, is a crop of the replicate-padded frame).

Per-layer checks feed each float64 reference layer with the kernel's OWN input map: act_{l-1} going forward, dact_l and
act_{l-1} going backward.  Layer 0's input is the fp32 `obs / 255.0 - 0.5` of the shifted frame, exactly the values
im2col_u8_aug's lookup table holds.  So every comparison holds exactly one layer of rounding and there is no ReLU flip
to excuse: the mask the reference applies is `act_{l-1} > 0` of the very map the kernel masked with.  Errors are rel-L2
over the whole map and, separately, the worst over frames, over the 2-pixel border band and over the 32 channels (an
error in one ragged quad of the N = 32 tile cannot hide in a norm); weight gradients also take the worst of the 9 taps
and of the 32 output channels.  Frames 0-3 take the extreme shifts (0, 0), (8, 8), (0, 8) and (8, 0), so every
replicate-clamped corner is reached.

Which kernels run depends on the precision and the batch (the coverage test at the end checks that all of them do):
- tf32, B % 4 == 0: layer 0 im2col_u8_aug + tensor-core GEMM (persistent from B ~ 46); layers 1-3 forward on the halo
  kernel (>= 592 tiles) or the conv_w GEMM + compact_grid; implicit weight gradient (scatter_to_grid with the bias
  column sums, one or four K-groups, diag_tap_sum); data gradient the implicit full correlation;
- tf32, B % 4 != 0: layers 1-3 forward as im2col_nhwc32 + GEMM, weight gradient as a plain GEMM (linear_wgrad);
- fp32: SIMT GEMMs throughout; folded weight gradient + diag_block_sum when B % 4 == 0; the no_grad forward and the
  data gradient run the SIMT conv_w GEMM + compact_grid.

Bars, about 3x the worst value measured on one NVIDIA B200 (1000 W power limit) over every case below, per slice:
- maps (act_l, dact_l, both forward paths): fp32 1e-6 (worst 3.6e-7: a channel of the no_grad forward's layer 2),
  tf32 2e-3 (worst 6.4e-4: a channel of the no_grad forward's layer 3 at B = 5; whole maps stay below 3.8e-4);
- weight gradients: fp32 2e-5 (worst 7.0e-6: a channel of dW_3 at C = 3, B = 256, a sum over 3.1e5 pixels),
  tf32 3e-3 (worst 9.8e-4: a channel of dW_1, all_active, C = 3, B = 5; whole tensors stay below 6.1e-4);
- bias gradients 2e-6 at either precision (worst 6.0e-7): they are summed in fp32 on CUDA cores.
Layouts and pitches are checked bit for bit.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

PAD = 36  # feature / gradient row pitch repr_dim + PAD, as the agents pass their wider LDE_ / F_ buffers
BAR = {"fp32": {"map": 1e-6, "dW": 2e-5, "db": 2e-6}, "tf32": {"map": 2e-3, "dW": 3e-3, "db": 2e-6}}
CHUNK = 256  # frames per float64 reference pass
EXTREME_SHIFTS = [[0, 0], [8, 8], [0, 8], [8, 0]]


# ------------------------------------------------------------------------------------------------ references
def input_map(obs, shifts):
    """Layer 0's input [B, C, H, H] fp32: the shift-augmented frame (a crop of the 4-pixel replicate-padded frame,
    shifts [B, 2] = (x, y) in [0, 8]) / 255 - 0.5.  The division is correctly rounded to fp32 (float64 then rounded:
    p / 255 repeats p's 8 bits, so it never lies on a rounding midpoint) and the subtraction is fp32, as in the kernel's
    lookup table and in the reference's `obs / 255.0 - 0.5`."""
    lut = (torch.arange(256, dtype=torch.float64, device=obs.device) / 255.0).float() - 0.5
    H = obs.shape[-1]
    p = F.pad(obs.float(), (4, 4, 4, 4), mode="replicate").long()
    crop = torch.stack([p[b, :, sy:sy + H, sx:sx + H] for b, (sx, sy) in enumerate(shifts.tolist())])
    return lut[crop]


def ref_layer(l, x, sd):
    """Pre-activation of layer l (`convnet.{2l}`) on a float64 NCHW map."""
    return F.conv2d(x, sd[f"convnet.{2 * l}.weight"], sd[f"convnet.{2 * l}.bias"], stride=2 if l == 0 else 1)


def chunks(B):
    return [(i, min(i + CHUNK, B)) for i in range(0, B, CHUNK)]


# ------------------------------------------------------------------------------------------------ error measures
def rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


def _worst(num, den):
    """max over slices of sqrt(num / den), slices with num == 0 counting as 0."""
    q = torch.where(num > 0, num.sqrt() / den.sqrt().clamp_min(1e-300), torch.zeros_like(num))
    return q.max().item()


def _worst_channel(num, den):
    """The worst channel, each measured against the larger of its own norm and the mean channel norm.  A channel the
    ReLU has nearly silenced, or a weight-gradient channel whose pixel sum nearly cancels (all_active: dW_l[o] ~
    mean(act) x sum_p dact_l[o, p] for every tap), has a norm far below the scale its rounding comes from; against its
    own norm alone plain rounding reads 1e-3 (tf32) to 3e-5 (fp32).  A wrong value in one channel still shows in full."""
    return _worst(num, torch.maximum(den, den.mean()))


def map_errors(out, ref):
    """rel-L2 over a [B, 32, h, h] map and the worst over frames, over the 2-pixel border band and over channels."""
    e = (out.double() - ref.double()) ** 2
    r = ref.double() ** 2
    H, W = out.shape[-2:]
    band = torch.ones(H, W, dtype=torch.bool, device=out.device)
    band[2:H - 2, 2:W - 2] = False
    return {"all": _worst(e.sum(), r.sum()),
            "frame": _worst(e.sum(dim=(1, 2, 3)), r.sum(dim=(1, 2, 3))),
            "border": _worst(e[..., band].sum(), r[..., band].sum()),
            "channel": _worst_channel(e.sum(dim=(0, 2, 3)), r.sum(dim=(0, 2, 3)))}


def weight_errors(out, ref):
    """rel-L2 over a [32, cin, 3, 3] weight gradient and the worst over the 9 taps and over the 32 output channels."""
    e = (out.double() - ref.double()) ** 2
    r = ref.double() ** 2
    return {"all": _worst(e.sum(), r.sum()),
            "tap": _worst(e.sum(dim=(0, 1)), r.sum(dim=(0, 1))),
            "channel": _worst_channel(e.sum(dim=(1, 2, 3)), r.sum(dim=(1, 2, 3)))}


def worst(errs):
    return max(v for e in errs.values() for v in e.values())


def fmt(errs):
    return ", ".join(f"{k} " + "/".join(f"{v:.1e}" for v in e.values()) for k, e in errs.items())


# ------------------------------------------------------------------------------------------------ fixtures
def make_params(channels, regime, seed):
    """He-scaled signed weights ("realistic"), or non-negative ones behind a +8 bias ("all_active": every
    pre-activation of the four layers is positive, so no ReLU mask is ever zero), as test_gpu_conv.py draws them."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for l, cin in enumerate((channels, 32, 32, 32)):
        w = torch.randn(32, cin, 3, 3, generator=g) * (2.0 / (cin * 9)) ** 0.5
        b = torch.randn(32, generator=g) * 0.1
        if regime == "all_active":
            w, b = (w.abs() / 8 if l > 0 else w), b + 8.0
        sd[f"convnet.{2 * l}.weight"], sd[f"convnet.{2 * l}.bias"] = w, b
    return sd


def make_inputs(channels, batch, height, seed):
    g = torch.Generator().manual_seed(seed)
    obs = torch.randint(0, 256, (batch, channels, height, height), generator=g, dtype=torch.uint8)
    shifts = torch.randint(0, 9, (batch, 2), generator=g, dtype=torch.int32)
    n = min(batch, 4)
    shifts[:n] = torch.tensor(EXTREME_SHIFTS[:n], dtype=torch.int32)
    return obs, shifts


def pitched(rows, fill):
    """rows [B, D] as a view of rows D + PAD wide whose padding columns hold `fill`; returns (full, view)."""
    full = torch.full((rows.shape[0], rows.shape[1] + PAD), fill, device="cuda")
    full[:, :rows.shape[1]] = rows.cuda()
    return full, full[:, :rows.shape[1]]


def make_encoder(channels, batch, height, precision, sd):
    from rlrep_b200.pixel import ConvEncoder
    enc = ConvEncoder((channels, height, height), batch=batch, precision=precision)
    enc.load_state_dict(sd)
    return enc


def forward_pitched(enc, obs, shifts, no_grad=False):
    """forward into a pitched feature buffer whose padding holds NaN; returns the full buffer."""
    feat_full, featv = pitched(torch.zeros(enc.batch, enc.repr_dim), float("nan"))
    enc.forward(obs.cuda(), shifts.cuda(), out=featv, no_grad=no_grad)
    torch.cuda.synchronize()
    return feat_full


def check_feat_layout(enc, feat_full):
    """The features are act_3 flattened in NCHW order, bit for bit; the padding columns are untouched."""
    D = enc.repr_dim
    act3 = enc.read_map("act", 3)
    assert torch.equal(feat_full[:, :D], act3.flatten(1)), "features differ from act_3"
    assert torch.isnan(feat_full[:, D:]).all(), "the forward wrote into the feature buffer's padding"
    return act3


def forward_errors(enc, sd64, obs, shifts, prefix="fwd"):
    """Per-layer forward errors of the handle's last forward; returns (errs, acts, x0)."""
    B = enc.batch
    x0 = input_map(obs.cuda(), shifts.cuda())
    acts = [enc.read_map("act", l) for l in range(4)]
    errs = {}
    for l in range(4):
        xin = x0 if l == 0 else acts[l - 1]
        ref = torch.cat([F.relu(ref_layer(l, xin[a:b].double(), sd64)) for a, b in chunks(B)])
        errs[f"{prefix}{l}"] = map_errors(acts[l], ref)
        del ref
    return errs, acts, x0


def backward_errors(enc, sd64, acts, x0):
    """Per-layer backward errors of the handle's last backward: dW_l, db_l and dact_{l-1} from the kernel's own dact_l
    and act_{l-1}."""
    B = enc.batch
    grads = enc.grads()
    dacts = [enc.read_map("dact", l) for l in range(4)]
    errs = {}
    for l in range(3, -1, -1):
        W = sd64[f"convnet.{2 * l}.weight"].clone().requires_grad_()
        bb = sd64[f"convnet.{2 * l}.bias"].clone().requires_grad_()
        dx_ref = []
        for a, b in chunks(B):
            xin = (x0 if l == 0 else acts[l - 1])[a:b].double().requires_grad_()
            y = ref_layer(l, xin, {f"convnet.{2 * l}.weight": W, f"convnet.{2 * l}.bias": bb})
            y.backward(dacts[l][a:b].double())
            if l > 0:
                dx_ref.append(xin.grad * (acts[l - 1][a:b] > 0))
        errs[f"dW{l}"] = weight_errors(grads[f"convnet.{2 * l}.weight"].cuda(), W.grad)
        errs[f"db{l}"] = {"all": rel(grads[f"convnet.{2 * l}.bias"].cuda(), bb.grad)}
        if l > 0:
            errs[f"dact{l - 1}"] = map_errors(dacts[l - 1], torch.cat(dx_ref))
        del dx_ref
    for k, v in grads.items():
        assert torch.isfinite(v).all(), k
    return errs, dacts


def assert_below_bar(errs, precision):
    def bar(key):
        return BAR[precision][key[:2] if key[:2] in ("dW", "db") else "map"]
    bad = {k: e for k, e in errs.items() if max(e.values()) >= bar(k)}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ per-layer tests
CASES = [(c, b, 84, prec, "realistic") for prec in ("fp32", "tf32")
         for c, b in ((9, 1), (9, 3), (9, 4), (9, 8), (9, 48), (9, 64), (9, 256), (3, 5), (3, 256))]
CASES += [(3, 1024, 84, "tf32", "realistic")]  # Latent Diff-SR encodes 4 x 256 frames per update
CASES += [(9, 8, 64, prec, "realistic") for prec in ("fp32", "tf32")]  # maps 31 / 29 / 27 / 25
CASES += [(c, b, 84, prec, "all_active") for prec in ("fp32", "tf32") for c, b in ((9, 4), (9, 48), (3, 5))]


@pytest.mark.parametrize("channels,batch,height,precision,regime", CASES)
def test_encoder_layers_match_float64(channels, batch, height, precision, regime):
    """Per-layer forward and backward: act_l, dW_l, db_l and dact_{l-1} = conv_transpose2d(dact_l, W_l) x (act_{l-1} > 0)
    against float64, through pitched feature and gradient buffers whose padding holds NaN.  The features must equal
    act_3 flattened bit for bit, and dact_3 must equal dfeat x (act_3 > 0) bit for bit."""
    seed = channels * 10000 + batch * 10 + height
    sd = make_params(channels, regime, seed)
    obs, shifts = make_inputs(channels, batch, height, seed + 1)
    dfeat = torch.randn(batch, 32 * ((height - 3) // 2 - 5) ** 2, generator=torch.Generator().manual_seed(seed + 2))
    enc = make_encoder(channels, batch, height, precision, sd)
    for k, v in enc.state_dict().items():
        assert torch.equal(v, sd[k]), k  # layout round trip through the C ABI
    assert dfeat.shape[1] == enc.repr_dim

    feat_full = forward_pitched(enc, obs, shifts)
    _, dfeatv = pitched(dfeat, float("nan"))
    enc.backward(dfeatv)
    torch.cuda.synchronize()

    sd64 = {k: v.double().cuda() for k, v in sd.items()}
    act3 = check_feat_layout(enc, feat_full)
    errs, acts, x0 = forward_errors(enc, sd64, obs, shifts)
    berrs, dacts = backward_errors(enc, sd64, acts, x0)
    errs.update(berrs)
    h3 = enc.hw(3)
    assert torch.equal(dacts[3], torch.where(act3 > 0, dfeat.cuda().view(batch, 32, h3, h3), torch.zeros_like(act3))), \
        "dact_3 differs from dfeat x (act_3 > 0)"
    for t in acts + dacts:
        assert torch.isfinite(t).all()
    print(f"\nC={channels} B={batch} H={height} {precision} {regime}: {fmt(errs)}")
    print(f"WORST C={channels} B={batch} H={height} {precision} {regime} {worst(errs):.3e}")
    assert_below_bar(errs, precision)
    enc.close()


# ------------------------------------------------------------------------------------------------ no_grad forward
NOGRAD_CASES = [(c, b, 84, prec) for prec in ("fp32", "tf32")
                for c, b in ((9, 1), (9, 3), (9, 4), (9, 8), (9, 48), (9, 256), (3, 5))]
NOGRAD_CASES += [(3, 768, 84, "tf32")]  # Latent Diff-SR's target forward over 3 x 256 frames
NOGRAD_CASES += [(9, 8, 64, prec) for prec in ("fp32", "tf32")]


@pytest.mark.parametrize("channels,batch,height,precision", NOGRAD_CASES)
def test_encoder_no_grad_forward(channels, batch, height, precision):
    """The evaluation-only forward (DrQ-v2's next-observation encoding) against the same float64 references, through a
    pitched feature buffer with NaN padding.  In fp32 and for batches that are not a multiple of 4 it runs another kernel
    chain than the forward with gradients; with tf32 and B % 4 == 0 both run valid_conv_3x3 and must agree bit for
    bit."""
    seed = 7000 + channels * 1000 + batch + height
    sd = make_params(channels, "realistic", seed)
    obs, shifts = make_inputs(channels, batch, height, seed + 1)
    enc = make_encoder(channels, batch, height, precision, sd)
    sd64 = {k: v.double().cuda() for k, v in sd.items()}

    feat_full = forward_pitched(enc, obs, shifts, no_grad=True)
    check_feat_layout(enc, feat_full)
    errs, acts, _ = forward_errors(enc, sd64, obs, shifts)
    for t in acts:
        assert torch.isfinite(t).all()
    print(f"\nno_grad C={channels} B={batch} H={height} {precision}: {fmt(errs)}")
    print(f"WORST no_grad C={channels} B={batch} H={height} {precision} {worst(errs):.3e}")
    assert_below_bar(errs, precision)

    if precision == "tf32" and batch % 4 == 0:
        feat_grad = forward_pitched(enc, obs, shifts)
        acts_grad = [enc.read_map("act", l) for l in range(4)]
        for l in range(4):
            assert torch.equal(acts_grad[l], acts[l]), f"act_{l}: no_grad and grad forward differ"
        assert torch.equal(feat_grad[:, :enc.repr_dim], feat_full[:, :enc.repr_dim])
    enc.close()


# ------------------------------------------------------------------------------------------------ state
@pytest.mark.parametrize("channels,batch,precision", [(9, 48, "tf32"), (9, 64, "tf32"), (9, 3, "tf32"), (3, 5, "fp32"),
                                                      (9, 8, "fp32")])
def test_encoder_deterministic_and_stateless(channels, batch, precision):
    """Two identical no_grad forward + forward + backward sequences give bit-identical features, maps and gradients, and
    a handle that first ran other weights and inputs gives results bit-identical to a fresh handle."""
    seed = 900 + channels * 100 + batch
    sd = make_params(channels, "realistic", seed)
    obs, shifts = make_inputs(channels, batch, 84, seed + 1)
    sd_o = make_params(channels, "all_active", seed + 2)
    obs_o, shifts_o = make_inputs(channels, batch, 84, seed + 3)
    dfeat = torch.randn(batch, 32 * 35 * 35, generator=torch.Generator().manual_seed(seed + 4)).cuda()

    def outputs(enc):
        enc.load_state_dict(sd)
        out = [forward_pitched(enc, obs_o, shifts, no_grad=True)[:, :enc.repr_dim]]
        out.append(forward_pitched(enc, obs, shifts)[:, :enc.repr_dim])
        enc.backward(dfeat)
        out += [enc.read_map(w, l) for w in ("act", "dact") for l in range(4)]
        return [t.cpu() for t in out] + list(enc.grads().values())

    used = make_encoder(channels, batch, 84, precision, sd_o)
    forward_pitched(used, obs_o, shifts_o)
    used.backward(dfeat * 3.0)
    forward_pitched(used, obs, shifts_o, no_grad=True)
    a, b = outputs(used), outputs(used)
    fresh = make_encoder(channels, batch, 84, precision, sd)
    c = outputs(fresh)
    for i, (u, v, w) in enumerate(zip(a, b, c)):
        assert torch.equal(u, v), f"output {i} differs between two identical calls"
        assert torch.equal(u, w), f"output {i} differs between a used and a fresh handle"
    used.close()
    fresh.close()


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_encoder_backward_refuses_stale_maps(precision):
    """backward() differentiates the maps of the last forward, so it must refuse after a forward that kept none for it
    (a no_grad forward, or none at all) instead of silently using another input's maps.  A refused call changes no
    gradient."""
    from rlrep_b200._lib import RlrepError
    B = 8
    sd = make_params(9, "realistic", 31)
    obs, shifts = make_inputs(9, B, 84, 32)
    dfeat = torch.randn(B, 32 * 35 * 35, generator=torch.Generator().manual_seed(33)).cuda()
    enc = make_encoder(9, B, 84, precision, sd)
    with pytest.raises(RlrepError, match="backward"):
        enc.backward(dfeat)
    forward_pitched(enc, obs, shifts)
    enc.backward(dfeat)
    grads = enc.grads()
    forward_pitched(enc, obs, shifts, no_grad=True)
    with pytest.raises(RlrepError, match="backward"):
        enc.backward(dfeat)
    _, dv = pitched(dfeat, float("nan"))
    with pytest.raises(RlrepError, match="backward"):
        enc.backward(dv)
    for k, v in enc.grads().items():
        assert torch.equal(v, grads[k]), k
    forward_pitched(enc, obs, shifts)  # a forward with gradients makes backward valid again, with the same result
    enc.backward(dfeat)
    enc.backward(dfeat)  # and stays valid: backward leaves the forward's maps as they are
    for k, v in enc.grads().items():
        assert torch.equal(v, grads[k]), k
    enc.close()


# ------------------------------------------------------------------------------------------------ coverage
def test_encoder_paths_are_reached():
    """The shapes of this file reach every encoder path: the uint8 im2col, the strided NHWC im2col, the tensor-core GEMM
    (persistent variant at B >= 48), the halo kernel, compaction after the conv_w GEMM, the SIMT GEMM, the implicit
    weight gradient's scatter and tap sum, the folded weight gradient's block sum and the layout kernels.  If the planner
    stops reaching one of them at these sizes, this test says so."""
    from torch.profiler import ProfilerActivity, profile
    names = set()
    for precision in ("fp32", "tf32"):
        for channels, batch in ((9, 3), (9, 8), (9, 48), (3, 64)):
            sd = make_params(channels, "realistic", channels + batch)
            obs, shifts = make_inputs(channels, batch, 84, channels + batch + 1)
            dfeat = torch.randn(batch, 32 * 35 * 35).cuda()
            enc = make_encoder(channels, batch, 84, precision, sd)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                forward_pitched(enc, obs, shifts, no_grad=True)
                forward_pitched(enc, obs, shifts)
                enc.backward(dfeat)
                torch.cuda.synchronize()
            names |= {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
            enc.close()
    want = ["im2col_u8_aug", "im2col_nhwc32", "gemm_tf32_kernel", "gemm_tf32_persistent", "gemm_conv_halo",
            "compact_grid", "gemm_tiled_kernel", "scatter_to_grid", "diag_tap_sum", "diag_block_sum", "pad_grid",
            "repack_flip", "nhwc_to_cp", "cp_to_nhwc"]
    missing = [w for w in want if not any(w in n for n in names)]
    print("\n" + "\n".join(sorted(n[:160] for n in names)))
    assert not missing, missing
