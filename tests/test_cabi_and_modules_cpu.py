"""CPU-only checks: the C-ABI library loads and exports exactly what include/pconv_b200.h declares, the module
mirror keeps the reference's state_dict surface, masks travel as HoleMask, and the product path refuses CPU
tensors instead of falling back."""
import json
import os
import re

import pytest
import torch

from conftest import ROOT

from text_segmentation_image_inpainting_b200 import _lib
from text_segmentation_image_inpainting_b200.masks import HoleMask
from text_segmentation_image_inpainting_b200.models import image_inpainting as PII
from text_segmentation_image_inpainting_b200.models import partial_convolution as PC


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "pconv_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(pcb_[a-z0-9_]+)\s*\(", txt)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/pconv_b200.h but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == syms, "ctypes signature table out of sync with the header"
    assert lib.pcb_version() == 1
    assert lib.pcb_launch_count() == 0 or lib.pcb_launch_count() > 0
    assert isinstance(lib.pcb_last_error(), bytes)


def test_argument_validation_without_gpu():
    """bad descriptors are rejected on the host, before any CUDA call"""
    lib = _lib.load()
    c = _lib.Conv()
    c.n = c.h = c.w = 8; c.cin = 4; c.cout = 4; c.kh = c.kw = 3; c.stride = 1; c.pad_h = c.pad_w = 1; c.dil = 1
    c.groups = 3; c.ho = c.wo = 8; c.nparts = 1; c.parts[0].c = 4; c.parts[0].x_cstride = 4
    rc = lib.pcb_pconv_forward(_lib.ctypes.byref(c), 1, None, 1, 4, 1, 1, None, None)
    assert rc != 0 and b"groups" in lib.pcb_last_error()
    c.groups = 1; c.ho = 7
    assert lib.pcb_pconv_forward(_lib.ctypes.byref(c), 1, None, 1, 4, 1, 1, None, None) != 0
    assert b"output size" in lib.pcb_last_error()
    assert lib.pcb_pconv_workspace(_lib.ctypes.byref(c)) == 0          # fp32 / 4 channels: generic path
    fe, de = _lib.c_size_t(0), _lib.c_size_t(0)
    c.ho = 8
    lib.pcb_conv_weight_layout(_lib.ctypes.byref(c), _lib.ctypes.byref(fe), _lib.ctypes.byref(de))
    assert (fe.value, de.value) == (4 * 9 * 4, 0)
    # a bf16 64->128 k3 layer is a tensor-core problem: K padded per tap, transposed copy for the data gradient
    c.dtype = _lib.PCB_BF16; c.cin = 64; c.cout = 128; c.parts[0].c = 64; c.parts[0].x_cstride = 64
    assert lib.pcb_conv_uses_tensor_cores(_lib.ctypes.byref(c)) == 1
    lib.pcb_conv_weight_layout(_lib.ctypes.byref(c), _lib.ctypes.byref(fe), _lib.ctypes.byref(de))
    assert (fe.value, de.value) == (128 * 9 * 64, 128 * 9 * 128)
    assert lib.pcb_pconv_workspace(_lib.ctypes.byref(c)) == 8 * 8 * 8 * 8
    # the RGB stem (3 channels in an 8-channel-padded NHWC buffer) runs row-packed: one K block per kernel row
    c.cin = 3; c.cout = 64; c.kh = c.kw = 7; c.pad_h = c.pad_w = 3; c.stride = 2; c.ho = c.wo = 4
    c.parts[0].c = 3; c.parts[0].x_cstride = 8
    assert lib.pcb_conv_uses_tensor_cores(_lib.ctypes.byref(c)) == 1
    lib.pcb_conv_weight_layout(_lib.ctypes.byref(c), _lib.ctypes.byref(fe), _lib.ctypes.byref(de))
    # row-packed operand, then the 4x4 space-to-depth problem of conv_stem.cu: 64 x (16 taps x 64-wide K blocks) bf16 + its fp32
    # staging 64 x 16 x 32 (two bf16 elements each)
    assert (fe.value, de.value) == (64 * 7 * 64 + 64 * 16 * 64 + 2 * 64 * 16 * 32, 0)
    c.parts[0].x_cstride = 3                                           # dense 3-channel pixels: not 16-byte chunks
    assert lib.pcb_conv_uses_tensor_cores(_lib.ctypes.byref(c)) == 0


def test_no_cpu_fallback():
    m = PC.PartialConv(4, 6, 3, 1, 1)
    with pytest.raises(_lib.PcbError):
        m((torch.zeros(1, 4, 8, 8), torch.ones(1, 4, 8, 8)))
    with pytest.raises(_lib.PcbError):
        PC.PartialActivatedBN(8, torch.nn.ReLU())((torch.zeros(1, 8, 4, 4), None))


def test_constructor_surface_and_state_dict_keys():
    pc = PC.PartialConv(4, 6, 3, 2, 1, 1, 1, True, same_holes=True)
    assert isinstance(pc.feature_conv, torch.nn.Conv2d) and pc.feature_conv.out_channels == 6
    sd = pc.state_dict()
    assert list(sd) == ["feature_conv.weight", "feature_conv.bias", "mask_conv.weight"]
    assert tuple(sd["mask_conv.weight"].shape) == (1, 1, 3, 3) and bool((sd["mask_conv.weight"] == 1).all())
    assert not pc.mask_conv.weight.requires_grad
    assert tuple(PC.PartialConv(4, 6, 3).state_dict()["mask_conv.weight"].shape) == (6, 4, 3, 3)
    with pytest.raises(AssertionError):
        PC.PartialConv1x1(4, 4, 3)
    with pytest.raises(AssertionError):
        PC.PartialConvNoHoles(4, 4, 3, groups=2)
    blk = PC.partial_convolution_block(4, 8, 3, 1, 1, activation=torch.nn.LeakyReLU(0.2))
    assert list(blk.state_dict()) == ["0.feature_conv.weight", "0.mask_conv.weight", "1.bn_act.0.weight", "1.bn_act.0.bias",
                                      "1.bn_act.0.running_mean", "1.bn_act.0.running_var", "1.bn_act.0.num_batches_tracked"]
    assert isinstance(PC.partial_convolution_block(4, 8, 1, use_1_conv=True, activation=None)[0], PC.PartialConv1x1)
    assert isinstance(PC.partial_convolution_block(4, 8, 1, no_holes_1_conv=True, activation=None)[0], PC.PartialConvNoHoles)
    with pytest.raises(TypeError):          # like the reference: the default activation=True is not an nn.Module
        PC.partial_convolution_block(4, 8, 3, 1, 1)
    assert isinstance(PC.partial_convolution_block(4, 8, 3, BN=False, activation=torch.nn.ReLU())[1], PC.PartialActivation)


def test_network_key_lists_match_reference_fixture():
    """tests/golden/state_dict_keys.json was written from the reference's own modules."""
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_keys.json")))
    from text_segmentation_image_inpainting_b200.models import text_segmentation as PTS
    assert set(ref) == {"ImageFillOrigin", "ImageFillOriginV2", "ImageFill", "TextSegament", "XceptionTextSegment"}
    for name, keys in ref.items():
        cls = getattr(PII, name, None) or getattr(PTS, name)
        mine = [[k, list(v.shape)] for k, v in cls().state_dict().items()]
        assert mine == keys, name


def test_lenient_load_state_dict_never_raises(capsys):
    net = PC.PartialConv(4, 6, 3)
    net.load_state_dict({"nope": torch.zeros(1), "feature_conv.weight": torch.zeros(9)})
    out = capsys.readouterr().out
    assert "is not in the model" in out and "fails to load" in out


def test_hole_mask_protocol():
    p = torch.ones(2, 4, 4, dtype=torch.uint8)
    m = HoleMask.from_plane(p, 3)
    assert tuple(m.shape) == (2, 3, 4, 4) and m.dtype == torch.float32 and isinstance(m, torch.Tensor)
    up = torch.nn.Upsample(scale_factor=2, mode="nearest")(m)
    assert isinstance(up, HoleMask) and tuple(up.shape) == (2, 3, 8, 8) and up.parts[0][2] == 1
    cat = torch.cat([up, HoleMask.from_plane(torch.ones(2, 8, 8, dtype=torch.uint8), 5)], dim=1)
    assert isinstance(cat, HoleMask) and tuple(cat.shape) == (2, 8, 8, 8) and [c for _, c, _ in cat.parts] == [3, 5]
    assert tuple(cat[:, :1].shape) == (2, 1, 8, 8)
    same = torch.cat([m, m], dim=1)
    assert len(same.parts) == 1 and same.parts[0][1] == 6          # adjacent identical planes merge
