"""Pins oracle/seg_torch.py (dense segmentation path) bit-for-bit against fixtures produced by the UNMODIFIED
reference (tests/golden/make_golden_seg.py).  CPU only."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import pconv_torch as OP
from oracle import seg_torch as O
from oracle.detfill import det_fill_state_dict, det_tensor

from conftest import GOLDEN

from text_segmentation_image_inpainting_b200.models import BaseModels as MB
from text_segmentation_image_inpainting_b200.models import MobileNetV2 as MM
from text_segmentation_image_inpainting_b200.models import common as MC
from text_segmentation_image_inpainting_b200.models import text_segmentation as MT

pytestmark = pytest.mark.usefixtures("golden_threads")

ACT = ("leaky", 0.3)


def _load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


def _sd(module):
    """key/shape skeleton from the product package's mirror, deterministically filled, trainable leaves"""
    return OP.clone_state_dict(det_fill_state_dict(module.state_dict()), requires_grad=True)


def _check(name, sd, fn):
    g = _load("seg_" + name)
    x = torch.from_numpy(g["x"]).requires_grad_(True)
    y = fn(sd, x)
    assert np.array_equal(y.detach().numpy(), g["y"]), name
    (y * torch.from_numpy(g["gy"])).sum().backward()
    assert np.array_equal(x.grad.numpy(), g["gx"]), name
    for k in [k for k in g if k.startswith("g.")]:
        assert np.array_equal(sd[k[2:]].grad.numpy(), g[k]), (name, k)
    for k in [k for k in g if k.startswith("bn.")]:
        assert np.array_equal(sd[k[3:]].numpy(), g[k]), (name, k)


def test_ds_conv_block():
    act = nn.LeakyReLU(0.3)
    _check("dsconv_s2", _sd(MB.DSConvBlock(16, 24, 3, 2, 1, 1, False, True, act, act)), lambda sd, x: O.ds_conv_block(sd, "", x, 3, 2, 1, 1, ACT, ACT))
    _check("dsconv_d4", _sd(MB.DSConvBlock(16, 16, 3, 1, 4, 4, False, True, act, None)), lambda sd, x: O.ds_conv_block(sd, "", x, 3, 1, 4, 4, ACT, None))


def test_inverted_residual_and_scse():
    act = nn.LeakyReLU(0.3)
    _check("invres_scse", _sd(MM.InvertedResidual(16, 16, 1, 6, 2, activation=act, bias=False, add_sece=True)),
           lambda sd, x: O.inverted_residual(sd, "", x, 16, 16, 1, 6, 2, ACT, True))
    _check("invres_s2", _sd(MM.InvertedResidual(16, 24, 2, 6, 1, activation=act, bias=False, add_sece=False)),
           lambda sd, x: O.inverted_residual(sd, "", x, 16, 24, 2, 6, 1, ACT, False))
    _check("scse", _sd(MC.SpatialChannelSqueezeExcitation(32, reduction=16, activation=act)), lambda sd, x: O.scse(sd, "", x, ACT))


def test_rfb_and_asp():
    act = nn.LeakyReLU(0.3)
    _check("rfb", _sd(MC.RFB(40, 16, activation=act, add_sece=True)), lambda sd, x: O.rfb(sd, "", x, 16, ACT, True))
    _check("asp", _sd(MC.ASP(24, 16, act, asp_rate=(3, 5, 9))), lambda sd, x: O.asp(sd, "", x, ACT, (3, 5, 9)))


@pytest.mark.parametrize("cls_name,tag", [("TextSegament", ""), ("XceptionTextSegment", ""),
                                          ("TextSegament", "_256"), ("XceptionTextSegment", "_256")])
def test_segmentation_network_forward_backward(cls_name, tag, capsys):
    g = _load("segnet_" + cls_name + tag)
    n, hw, step = int(g["n"]), int(g["hw"]), int(g["step"])
    sd = _sd(getattr(MT, cls_name)())
    x = det_tensor(cls_name + ".x", (n, 3, hw, hw))
    out = O.NETWORKS[cls_name](sd, x)
    assert np.array_equal(out[..., ::step, ::step].detach().numpy(), g["out_sub"])
    assert np.array_equal(out[0, :, hw // 2, :].detach().numpy(), g["out_row"])
    loss = out.abs().mean()
    assert float(loss.detach()) == float(g["loss"])
    loss.backward()
    for k in [k for k in g if k.startswith("g.")]:
        assert np.array_equal(sd[k[2:]].grad.numpy(), g[k]), k
    for k in [k for k in g if k.startswith("bn.")]:
        assert np.array_equal(sd[k[3:]].numpy(), g[k]), k
