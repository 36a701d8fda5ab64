"""CPU suite: host-side logic -- graph configs, module/state_dict mirror, planner, C-ABI exports,
drop-in install/convert into the reference namespace, and "fails loudly without CUDA"."""
import ctypes
import json
import os
import re

import pytest
import torch

from oracle import ref_shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", ["yolov5l_fusion_transformerx3_FLIR_aligned", "yolov5l_fusion_transformerx3_llvip",
                                  "yolov5s_fusion_transformerx3_vedai"])
def test_generated_config_equals_reference_yaml(name, cft, golden_dir):
    """``yaml.safe_load`` of the reference's graph files, stored by oracle/make_golden.py."""
    with open(os.path.join(golden_dir, "reference_x3_yaml.json")) as f:
        assert json.load(f)[name] == cft.named_config(name)


@pytest.mark.parametrize("name,nkeys,nparams", [
    ("yolov5s_fusion_transformerx3_vedai", 965, 44.54e6),
    ("yolov5l_fusion_transformerx3_FLIR_aligned", 1445, 206.26e6),
    ("yolov5x_fusion_transformerx3_FLIR_aligned", 1685, 344.52e6),
])
def test_model_state_dict_mirrors_reference(name, nkeys, nparams, cft, oracle):
    cfg = cft.named_config(name)
    model = cft.Model(cfg)
    sd = oracle.init_state(cfg)                      # reference key names (pinned by make_golden.py)
    msd = model.state_dict()
    assert len(msd) == nkeys and set(msd) == set(sd)
    assert all(msd[k].shape == sd[k].shape for k in sd)
    model.load_state_dict(sd, strict=True)
    n = sum(p.numel() for p in model.parameters())
    assert abs(n - nparams) / nparams < 1e-3
    assert [m.i for m in model.model] == list(range(47))
    det = model.model[-1]
    assert det.stride.tolist() == [8.0, 16.0, 32.0] and det.no == cfg["nc"] + 5
    assert torch.allclose(det.anchors * det.stride.view(-1, 1, 1), det.anchor_grid.view(3, 3, 2))


def test_planner_finds_concat_slots_and_gpt_groups(cft):
    model = cft.Model(cft.named_config("yolov5l_fusion_transformerx3_FLIR_aligned"))
    plan = model._plan
    assert plan["gpt_groups"] == {10: {"rgb": 11, "ir": 12, "sum": 29}, 17: {"rgb": 18, "ir": 19, "sum": 30},
                                  26: {"rgb": 27, "ir": 28, "sum": 31}}
    assert plan["slots"][33][:4] == (34, 0, 512, 1024) and plan["slots"][30][:4] == (34, 512, 1024, 1024)
    assert plan["slots"][32][:4] == (44, 512, 1024, 1024) and plan["slots"][36][:4] == (41, 256, 512, 512)
    assert sorted(set(model.save)) == [1, 4, 9, 10, 11, 12, 14, 16, 17, 18, 19, 22, 25, 26, 27, 28, 29, 30, 32, 36, 39, 42, 45]
    # the producer's scale relative to its own input sizes the Concat buffer: Upsample doubles, Conv stride 2 halves
    assert plan["slots"][33][4] == (2, 1) and plan["slots"][30][4] == (1, 1)
    strided = [i for i, sl in plan["slots"].items() if sl[4] == (1, 2)]
    assert strided and all(isinstance(model.model[i], cft.modules.Conv) and model.model[i].conv.stride[0] == 2 for i in strided)


def test_planner_sizes_concat_buffers_from_the_stride_table(cft):
    """A Focus (or any resolution-changing producer) writing into a Concat gets a buffer of its OUTPUT resolution; producers
    at different total strides are not planned into one buffer (ADVICE r1: `_slot()` looked at Upsample / Conv only)."""
    from importlib import import_module
    model_mod = import_module(cft.__name__ + ".model")
    M = cft.modules

    def layer(m, i, f):
        m.i, m.f = i, f
        return m
    import torch.nn as nn
    layers = nn.Sequential(layer(M.Focus(3, 16, 3), 0, -1), layer(M.Focus(3, 16, 3), 1, -4), layer(M.Concat(1), 2, [0, 1]),
                           layer(M.Conv(32, 32, 3, 2), 3, -1), layer(M.Concat(1), 4, [2, 3]))
    plan = model_mod._plan_graph(layers)
    assert plan["slots"][0] == (2, 0, 16, 32, (1, 2)) and plan["slots"][1] == (2, 16, 32, 32, (1, 2))
    assert 3 not in plan["slots"] and 2 not in plan["slots"]          # stride 2 vs stride 4: never one buffer


def test_c_abi_exports_every_declared_symbol(cft):
    header = open(os.path.join(ROOT, "include", "cft_b200.h")).read()
    declared = set(re.findall(r"\b(cft_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 18
    lib = cft.load()                                   # dlopen only; no device work
    for name in declared:
        assert hasattr(lib, name), f"libcft_b200.so does not export {name}"
    assert set(cft._lib.SIGNATURES) == declared
    assert lib.cft_abi_version() == 7


def test_forward_fails_loudly_without_cuda(cft):
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    model = cft.Model(cft.named_config("yolov5s_fusion_transformerx3_vedai")).eval()
    x = torch.rand(1, 3, 64, 64)
    with pytest.raises(cft.CftError):
        model(x, x)


def test_attention_rejects_misaligned_pointers(cft):
    """Both attention kernels move q / k / v and the output in 16-byte vectors, so cft_attention refuses a qkv or out
    pointer that is not 16-byte aligned (CFT_E_ARG) before it touches the device.  The pointers are fake: without a
    GPU the call can only return an error; with one, an unchecked build would dereference them."""
    if torch.cuda.is_available():
        pytest.skip("fake device pointers: run only where no kernel can be launched")
    lib = cft.load()
    good_qkv, good_out = 0x10000000, 0x20000000
    for qkv, out in ((good_qkv + 2, good_out), (good_qkv + 8, good_out), (good_qkv, good_out + 2),
                     (good_qkv, good_out + 8), (good_qkv + 4, good_out + 4)):
        for T, dk in ((128, 64), (64, 8)):                              # the tcgen05 shape and a CUDA-core-only one
            rc = lib.cft_attention(qkv, out, 2, T, 8 * dk, 8, None)
            assert rc == 1, (hex(qkv), hex(out), T, rc)                 # CFT_E_ARG
            assert "aligned" in lib.cft_last_error().decode()


def test_weight_packing_folds_bn_like_reference(cft):
    """pack_conv_weight == fuse_conv_and_bn (utils/torch_utils.py:181-201) then OIHW -> [O][tap][I]."""
    from importlib import import_module
    model_mod = import_module("multispectral-object-detection_b200.model")
    torch.manual_seed(0)
    conv = cft.Conv(16, 24, 3, 1)
    conv.bn.eps = 1e-3
    conv.bn.weight.data.uniform_(0.5, 1.5); conv.bn.bias.data.normal_(0, .1)
    conv.bn.running_mean.normal_(0, .1); conv.bn.running_var.uniform_(.5, 1.5)
    fused = model_mod.fuse_conv_and_bn(conv.conv, conv.bn)
    w, b = cft.ops.pack_conv_weight(conv.conv.weight, None, (conv.bn.weight, conv.bn.bias, conv.bn.running_mean,
                                                              conv.bn.running_var, conv.bn.eps))
    ref = fused.weight.detach().permute(0, 2, 3, 1).reshape(24, 9, 16)
    assert w.shape == (24, 9, 16) and w.dtype == torch.bfloat16
    assert (w.float() - ref).abs().max() <= ref.abs().max() * 2 ** -8
    assert torch.allclose(b, fused.bias.detach(), atol=1e-6)


@pytest.mark.skipif(not ref_shim.available(), reason="needs the reference project's own Python modules")
def test_install_and_convert_into_reference(cft, oracle):
    yt = ref_shim.import_reference()
    name = "yolov5s_fusion_transformerx3_vedai"
    cfg = cft.named_config(name)
    sd = oracle.init_state(cfg)
    prev = cft.install(yt)
    try:
        rm = yt.Model(ref_shim.reference_yaml(name), ch=3).eval()      # the reference's own Model/parse_model
    finally:
        cft.uninstall(yt, prev)
    mods = {type(m).__module__ for m in rm.model}
    assert mods == {"multispectral-object-detection_b200.modules"}
    rm.load_state_dict(sd, strict=True)
    assert sorted(set(rm.save)) == sorted(set(cft.Model(cfg).save))
    # convert(): an already-built reference model keeps its weights
    rm2 = yt.Model(ref_shim.reference_yaml(name), ch=3).eval()
    assert type(rm2.model[0]).__module__ == "models.common"
    rm2.load_state_dict(sd, strict=True)
    rm3 = cft.convert(rm2)
    sd3 = rm3.state_dict()
    assert set(sd3) == set(sd) and all(torch.equal(sd3[k], sd[k]) for k in sd)
    assert all(type(m).__module__ == "multispectral-object-detection_b200.modules" for m in rm3.model)


def test_focus_weight_reindexing_is_a_6x6_stride2_conv(cft):
    """pack_focus_weight: Focus (space-to-depth + 3x3 / pad 1, models/common.py:168-180) == 6x6 / stride 2 / pad 2 conv
    on the image with the re-indexed filter (the identity the fused CUDA kernel is built on), checked in fp64 on CPU."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(0)
    w = torch.randn(16, 12, 3, 3, generator=g)
    b = torch.randn(16, generator=g)
    x = torch.rand(2, 3, 20, 28, generator=g)
    s2d = torch.cat([x[..., ::2, ::2], x[..., 1::2, ::2], x[..., ::2, 1::2], x[..., 1::2, 1::2]], 1)
    ref = F.conv2d(s2d.double(), w.double(), b.double(), padding=1)
    wf, bf = cft.ops.pack_focus_weight(w, b, None, device="cpu")
    assert wf.shape == (16, 192) and wf.dtype == torch.float16 and torch.equal(bf, b)
    w6 = wf.float().view(16, 24, 8)
    assert (w6[:, 18:] == 0).all() and (w6[:, :, 6:] == 0).all()
    k66 = w.view(16, 2, 2, 3, 3, 3).permute(0, 3, 4, 2, 5, 1).reshape(16, 3, 6, 6)      # exact (unrounded) 6x6 filter
    assert torch.allclose(w6[:, :18, :6].reshape(16, 3, 6, 6), k66, atol=2e-3, rtol=1e-3)   # fp16 rounding only
    y = F.conv2d(x.double(), k66.double(), b.double(), stride=2, padding=2)
    assert y.shape == ref.shape and torch.allclose(y, ref, atol=1e-12)


def test_product_package_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under the package directory may import or execute it (no CPU fallback,
    no checker on the product path)."""
    pkg_dir = os.path.join(ROOT, "multispectral-object-detection_b200")
    offenders = []
    for dirpath, _, files in os.walk(pkg_dir):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, fn), errors="ignore").read()
                if re.search(r"^\s*(from|import)\s+oracle\b", text, re.M) or "oracle/" in text or "cft_oracle" in text:
                    offenders.append(os.path.join(dirpath, fn))
    assert not offenders, offenders


def test_training_mode_batchnorm_fails_loudly(cft):
    """The forward folds BN running statistics (eval semantics); a train-mode BatchNorm must raise, not silently run eval."""
    conv = cft.Conv(16, 24, 3, 1)
    assert conv.training
    with pytest.raises(cft.CftError, match="training mode"):
        conv.folded("cpu")
    conv.eval()
    w, b = conv.folded("cpu")
    assert w.shape == (24, 9, 16)
    c3 = cft.C3(16, 16, 1)
    with pytest.raises(cft.CftError, match="training mode"):
        c3._cv12("cpu")


def test_convert_keeps_batchnorm_eps_numeric(cft):
    """ADVICE r1: ``convert()`` must fold BatchNorm with the SOURCE module's eps (the reference sets 1e-3,
    utils/torch_utils.py:144-153; a fresh nn.BatchNorm2d has 1e-5) -- checked on the folded weights of an unfused Conv with
    small running variances, where the two eps values differ by up to 40 %."""
    from importlib import import_module
    M = import_module("multispectral-object-detection_b200.modules")
    model_mod = import_module("multispectral-object-detection_b200.model")
    torch.manual_seed(0)
    src = M.Conv(16, 32, 3, 1).eval()
    src.bn.eps, src.bn.momentum = 1e-3, 0.03
    with torch.no_grad():
        src.bn.running_var.uniform_(1e-4, 2e-3)
        src.bn.running_mean.normal_(0, 0.1)
        src.bn.weight.uniform_(0.5, 1.5)
        src.bn.bias.normal_(0, 0.1)
    new = model_mod._convert_module(src)
    assert new.bn.eps == 1e-3 and new.bn.momentum == 0.03 and not new.training
    w, b = new.folded(torch.device("cpu"))
    scale = src.bn.weight / torch.sqrt(src.bn.running_var + 1e-3)            # utils/torch_utils.py:181-201
    w_ref = (src.conv.weight * scale.view(-1, 1, 1, 1)).permute(0, 2, 3, 1).reshape(32, 9, 16)
    b_ref = src.bn.bias - src.bn.running_mean * scale
    assert torch.allclose(w.float(), w_ref.detach().to(torch.bfloat16).float(), atol=0, rtol=0)
    assert torch.allclose(b, b_ref.detach(), atol=1e-6)
    wrong = src.bn.weight / torch.sqrt(src.bn.running_var + 1e-5)
    assert float((wrong / scale).max()) > 1.2                                # the test can tell the two eps apart


def test_c3_and_gpt_refuse_training_mode(cft):
    """Eval-only forward: a C3 whose cv1|cv2 weights are already packed, and a GPT with dropout, fail loudly in train mode."""
    from importlib import import_module
    M = import_module("multispectral-object-detection_b200.modules")
    c3 = M.C3(32, 32, 1).train()
    with pytest.raises(cft.CftError):
        M._require_eval_bn(c3.cv1.bn)
    g = M.GPT(64, n_layer=1).train()
    with pytest.raises(cft.CftError):
        g.tokens(torch.zeros(1, 64, 8, 8), torch.zeros(1, 64, 8, 8))
