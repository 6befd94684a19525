"""Pins the oracle (oracle/pconv_torch.py, oracle/pconv_box.c) against golden fixtures produced
by the UNMODIFIED reference (tests/golden/make_golden.py).  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import pconv_torch as O
from oracle.detfill import det_fill_state_dict, det_tensor
from oracle.pconv_box import pconv_box_forward

from conftest import GOLDEN

pytestmark = pytest.mark.usefixtures("golden_threads")

L1 = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "pc_*.npz")))


def _load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


def _t(a):
    return torch.from_numpy(np.array(a))


def _run_l1(name, g, requires_grad=False):
    cin, cout, k, s, p, d, groups, bias, sh = [int(v) for v in g["cfg"]]
    x = _t(g["x"]).requires_grad_(requires_grad)
    w = _t(g["sd.feature_conv.weight"]).requires_grad_(requires_grad)
    b = _t(g["sd.feature_conv.bias"]).requires_grad_(requires_grad) if bias else None
    mask = _t(g["mask"])
    if name.startswith("pc_1x1"):
        y, nm = O.partial_conv_1x1(x, mask, w, b, groups)
    elif name.startswith("pc_noholes"):
        y, nm = O.partial_conv_no_holes(x, mask, w, b, s, p, d)
    else:
        y, nm = O.partial_conv(x, mask, w, b, s, p, d, groups, bool(sh))
    return x, w, b, y, nm


@pytest.mark.parametrize("name", L1)
def test_l1_forward_bit_exact(name):
    g = _load(name)
    _, _, _, y, nm = _run_l1(name, g)
    assert np.array_equal(y.detach().numpy(), g["y"], equal_nan=True)
    assert np.array_equal(nm.contiguous().numpy(), g["new_mask"])


@pytest.mark.parametrize("name", L1)
def test_l1_backward_bit_exact(name):
    g = _load(name)
    x, w, b, y, _ = _run_l1(name, g, requires_grad=True)
    gy = _t(g["gy"])
    (torch.where(torch.isfinite(y), y, torch.zeros_like(y)) * gy).sum().backward()
    assert np.array_equal(x.grad.numpy(), g["gx"], equal_nan=True)
    assert np.array_equal(w.grad.numpy(), g["gw"], equal_nan=True)
    if b is not None:
        assert np.array_equal(b.grad.numpy(), g["gb"], equal_nan=True)


@pytest.mark.parametrize("name", [n for n in L1 if not n.startswith(("pc_1x1", "pc_noholes"))])
def test_c_box_sum_restatement(name):
    """plain-C direct-loop / box-sum restatement: masks bit-exact, features to 1e-5."""
    g = _load(name)
    cin, cout, k, s, p, d, groups, bias, sh = [int(v) for v in g["cfg"]]
    y, ms, nm = pconv_box_forward(g["x"], g["mask"], g["sd.feature_conv.weight"],
                                  g["sd.feature_conv.bias"] if bias else None, s, p, d, groups, bool(sh))
    assert np.array_equal(nm, g["new_mask"])
    scale = np.abs(g["y"]).max()
    assert np.abs(y - g["y"]).max() <= 1e-5 * scale


def test_documented_behaviours():
    """SURVEY 8c: hole interior -> y==0 & m'==0; a 32x32 hole under k3 p1 leaves a 30x30 hole;
    same_holes == full-mask path for channel-uniform masks; NoHoles NaNs on an all-hole window."""
    x = det_tensor("beh.x", (1, 4, 48, 48)); mask = torch.ones_like(x); mask[:, :, 8:40, 8:40] = 0
    w = det_tensor("beh.w", (6, 4, 3, 3), scale=0.2); b = det_tensor("beh.b", (6,), scale=0.1)
    y, nm = O.partial_conv(x, mask, w, b, 1, 1, 1, 1, False)
    assert int((nm[0, 0] == 0).sum()) == 30 * 30
    assert torch.all(y[nm == 0] == 0)
    y2, nm2 = O.partial_conv(x, mask, w, b, 1, 1, 1, 1, True)
    assert torch.equal(y, y2) and torch.equal(nm, nm2.contiguous())
    y3, _ = O.partial_conv_no_holes(x, mask, w, b, 1, 1, 1)
    assert torch.isnan(y3[0, 0, 20, 20])
    # depthwise + same_holes divides by count * in_channels (reference quirk)
    wd = det_tensor("beh.wd", (4, 1, 3, 3)); ones = torch.ones_like(x)
    yd, _ = O.partial_conv(x, ones, wd, None, 1, 1, 1, 4, True)
    plain = torch.nn.functional.conv2d(x, wd, None, 1, 1, 1, 4)
    assert torch.allclose(yd[0, :, 5, 5] * 36.0, plain[0, :, 5, 5], rtol=1e-5, atol=1e-6)


def test_block_bn_running_stats():
    g = _load("block_bn_leaky")
    sd = {k[4:]: _t(v).clone() for k, v in g.items() if k.startswith("sd0.")}
    for k in sd:
        if sd[k].is_floating_point() and not k.endswith(("running_mean", "running_var", "mask_conv.weight")):
            sd[k].requires_grad_(True)
    x = _t(g["x"]).requires_grad_(True); mask = _t(g["mask"])
    kw = dict(k=3, s=2, p=1, bn=True, act=("leaky", 0.2), same_holes=True)
    y1, m1 = O.pconv_block(sd, "", x, mask, training=True, **kw)
    assert np.array_equal(y1.detach().numpy(), g["y1"]) and np.array_equal(m1.contiguous().numpy(), g["m1"])
    (y1 * _t(g["gy"])).sum().backward()
    assert np.array_equal(x.grad.numpy(), g["gx"])
    for k in ("0.feature_conv.weight", "1.bn_act.0.weight", "1.bn_act.0.bias"):
        assert np.array_equal(sd[k].grad.numpy(), g["g." + k]), k
    with torch.no_grad():
        y2, _ = O.pconv_block(sd, "", x.detach() * 0.5 + 0.25, mask, training=True, **kw)
        assert np.array_equal(y2.numpy(), g["y2"])
        for k in ("1.bn_act.0.running_mean", "1.bn_act.0.running_var", "1.bn_act.0.num_batches_tracked"):
            assert np.array_equal(sd[k].numpy(), g["sd2." + k]), k
        y3, _ = O.pconv_block(sd, "", x.detach(), mask, training=False, **kw)
        assert np.array_equal(y3.numpy(), g["y3"])


def test_double_upsample():
    g = _load("double_upsample")
    xu, mu = O.double_upsample(_t(g["x"]), _t(g["mask"]))
    assert np.array_equal(xu.numpy(), g["xu"]) and np.array_equal(mu.numpy(), g["mu"])


def _net_state_dict(cls_name):
    """Key/shape skeleton of the reference network, rebuilt from the product package's own mirror
    (so this test does not need /root/reference), then deterministically filled."""
    from text_segmentation_image_inpainting_b200.models import image_inpainting as pii
    with torch.device("cpu"):
        net = getattr(pii, cls_name)()
    return det_fill_state_dict(net.state_dict())


@pytest.mark.parametrize("cls_name,tag", [("ImageFillOrigin", ""), ("ImageFillOriginV2", ""), ("ImageFill", ""),
                                          ("ImageFillOrigin", "_512")])      # _512: the benchmarked resolution
def test_network_forward_backward(cls_name, tag):
    g = _load("net_" + cls_name + tag)
    n, hw, step = int(g["n"]), int(g["hw"]), int(g["step"])
    sd = O.clone_state_dict(_net_state_dict(cls_name), requires_grad=True)
    plane = np.unpackbits(g["mask_bits"])[: n * hw * hw].reshape(n, 1, hw, hw).astype(np.float32)
    mask = torch.from_numpy(np.repeat(plane, 3, 1))
    x = det_tensor(cls_name + ".x", (n, 3, hw, hw))
    out = O.NETWORKS[cls_name](sd, x * mask, mask, training=True)
    assert np.array_equal(out[..., ::step, ::step].detach().numpy(), g["out_sub"])
    assert np.array_equal(out[0, :, hw // 2, :].detach().numpy(), g["out_row"])
    loss = out.abs().mean()
    assert float(loss) == float(g["loss"])
    loss.backward()
    for k in [k for k in g if k.startswith("g.")]:
        assert np.array_equal(sd[k[2:]].grad.numpy(), g[k]), k
    for k in [k for k in g if k.startswith("gsum.")]:
        got = float(sd[k[5:]].grad.double().abs().sum())
        assert abs(got - float(g[k])) <= 1e-9 * max(1.0, abs(float(g[k]))), k
    for k in [k for k in g if k.startswith("bn.")]:
        assert np.array_equal(sd[k[3:]].numpy(), g[k]), k


def test_bf16_storage_emulation_is_off_by_default_and_documents_the_precision_gap():
    """oracle.pconv_torch.storage(bfloat16) rounds activations / activation gradients where the CUDA path's tensor-core mode
    stores them in bf16.  (a) Outside the context manager the oracle is untouched (the golden tests above pin that bit for bit);
    (b) under it the forward stays within bf16 rounding of the fp32 reference while gradients that pass through a BatchNorm move
    by far more than bf16 epsilon on ill-conditioned channels -- the reason the GPU parity tests compare bf16 gradients with the
    emulated oracle and only the forward / loss / tail layer with the fp32 reference."""
    cls_name, n, hw = "ImageFillOrigin", 2, 256
    sd0 = _net_state_dict(cls_name)
    x = det_tensor("emu.x", (n, 3, hw, hw))
    from text_segmentation_image_inpainting_b200.synthetic import random_hole_masks
    mask = torch.from_numpy(random_hole_masks(n, hw, hw, seed=3))

    def run(st):
        sd = O.clone_state_dict(sd0, requires_grad=True)
        with O.storage(st):
            xin = x * mask if st is None else (x * mask).to(st).float()
            out = O.NETWORKS[cls_name](sd, xin, mask, training=True)
            if st is not None:
                out = O._rb(O._rf(out))
            loss = out.abs().mean()
            loss.backward()
        return out.detach(), float(loss.detach()), {k: v.grad for k, v in sd.items() if v.grad is not None}

    assert O._STORAGE is None
    o32, l32, g32 = run(None)
    o16, l16, g16 = run(torch.bfloat16)
    assert O._STORAGE is None
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())  # noqa: E731
    assert rel(o16, o32) <= 2e-2 and abs(l16 - l32) <= 2e-3 * l32
    assert rel(g16["decoder.7.0.feature_conv.weight"], g32["decoder.7.0.feature_conv.weight"]) <= 1e-2      # no BatchNorm behind it
    gap = max(rel(g16[k], g32[k]) for k in g32 if ".bn_act." in k or k.startswith("decoder.6.0.0"))
    assert gap > 2e-2, gap            # the gap this emulation exists to account for
