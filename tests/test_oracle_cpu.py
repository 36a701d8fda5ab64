"""CPU suite (-m "not gpu"): the oracle against the committed golden vectors (which are outputs of the
UNMODIFIED reference, see oracle/make_golden.py)."""
import glob
import os

import pytest
import torch


def _cases(golden_dir):
    return sorted(glob.glob(os.path.join(golden_dir, "*.pt")))


def test_golden_files_present(golden_dir):
    assert len(_cases(golden_dir)) >= 5


@pytest.mark.parametrize("name", ["s_vedai_b2_128x160", "s_vedai_b1_64x64_fused", "l_flir_b1_64x64",
                                  "l_llvip_b1_64x96", "x_flir_b1_64x64"])
def test_oracle_matches_reference_golden(name, golden_dir, cft, oracle):
    g = torch.load(os.path.join(golden_dir, name + ".pt"))
    cfg = cft.named_config(g["config"])
    sd = oracle.init_state(cfg, seed=g["weight_seed"])
    x, x2 = oracle.make_inputs(g["batch"], g["height"], g["width"], seed=g["input_seed"])
    # the seeded generators must reproduce the tensors the reference saw
    assert abs(float(x.double().sum()) - g["input_checksum"][0]) < 1e-6
    assert abs(float(x2.double().sum()) - g["input_checksum"][1]) < 1e-6
    assert abs(float(sum(v.double().abs().sum() for v in sd.values())) - g["state_checksum"]) < 1e-3
    if g["fused"]:
        sd = fuse_state(sd)
    z, raw = oracle.forward(sd, cfg, x, x2)
    assert z.shape == g["z"].shape
    # fp32 CPU: identical op sequence -> tight; fused goldens differ by the fold's rounding only
    tol = 2e-3 if g["fused"] else 1e-4
    assert_close_fp32(z[..., :4], g["z"][..., :4], tol)                  # boxes, in pixels
    assert_close_fp32(z[..., 4:], g["z"][..., 4:], tol)                  # scores
    for a, b in zip(raw, g["raw"]):
        assert_close_fp32(a, b, 1e-3 if g["fused"] else 1e-5)


def assert_close_fp32(a, b, atol):
    """max|a - b| <= atol + 64 fp32 eps x max|b|.  The goldens were written with 8 intra-op threads and the oracle
    reproduces them exactly at that count; PyTorch's CPU kernels split their fp32 sums by thread count, so another count
    (``torch.set_num_threads`` 1, 4 or 16, on the same AVX-512 host) differs by up to 26 eps of the tensor's largest value
    in the z boxes (l_flir_b1_64x64) and 20 eps in the raw heads."""
    assert (a - b).abs().max().item() <= atol + 64 * torch.finfo(torch.float32).eps * b.abs().max().item()


def fuse_state(sd):
    """BN folding of utils/torch_utils.py:181-201 applied to a flat state dict."""
    out = {}
    for k, v in sd.items():
        if k.endswith("conv.weight") and k[:-len("conv.weight")] + "bn.weight" in sd:
            p = k[:-len("conv.weight")]
            scale = sd[p + "bn.weight"] / torch.sqrt(sd[p + "bn.running_var"] + 1e-3)
            out[k] = v * scale.view(-1, 1, 1, 1)
            out[p + "conv.bias"] = sd[p + "bn.bias"] - sd[p + "bn.running_mean"] * scale
        elif ".bn." in k:
            continue
        else:
            out[k] = v
    return out


def test_detect_grid_and_row_order(oracle):
    """models/yolo_test.py:48-64: flat row = a*ny*nx + j*nx + i, grid = (i, j), levels P3,P4,P5."""
    na, no = 3, 8
    raw = [torch.zeros(1, na, ny, nx, no) for ny, nx in ((4, 6), (2, 3), (1, 2))]
    ag = torch.tensor([[10, 13, 16, 30, 33, 23], [30, 61, 62, 45, 59, 119], [116, 90, 156, 198, 373, 326]]).float().view(3, 1, 3, 1, 1, 2)
    z = oracle.decode_heads(raw, ag)
    assert z.shape == (1, 3 * (24 + 6 + 2), no)
    # sigmoid(0) = .5 -> xy = (0.5 + grid) * stride ; wh = anchor
    row = 1 * 24 + 2 * 6 + 5          # level 0, anchor 1, j=2, i=5
    assert z[0, row, 0].item() == (0.5 + 5) * 8 and z[0, row, 1].item() == (0.5 + 2) * 8
    assert z[0, row, 2].item() == 16 and z[0, row, 3].item() == 30
    row = 3 * 24 + 2 * 6 + 1 * 3 + 2  # level 1, anchor 2, j=1, i=2
    assert z[0, row, 0].item() == (0.5 + 2) * 16 and z[0, row, 1].item() == (0.5 + 1) * 16
    assert z[0, row, 2].item() == 59 and z[0, row, 3].item() == 119


def test_flop_model(cft, oracle):
    """SURVEY.md §8(d): 224.38 GFLOP/pair (l@640), 36.15 (s@640), 414.90 (x@640), 641.42 (l@1024x1280)."""
    f = oracle.conv_linear_flops
    assert abs(f(cft.named_config("yolov5l_fusion_transformerx3_FLIR_aligned"), 640, 640) / 1e9 - 224.38) < 0.01
    assert abs(f(cft.named_config("yolov5s_fusion_transformerx3_vedai"), 640, 640) / 1e9 - 36.15) < 0.01
    assert abs(f(cft.named_config("yolov5x_fusion_transformerx3_FLIR_aligned"), 640, 640) / 1e9 - 414.90) < 0.01
    assert abs(f(cft.named_config("yolov5l_fusion_transformerx3_llvip"), 1024, 1280) / 1e9 - 641.42) < 0.01


def test_oracle_equals_stored_reference(golden_dir, cft, oracle):
    """The reference's own eval forward (s graph, weight seed 11, input seed 12), stored by oracle/make_golden.py."""
    g = torch.load(os.path.join(golden_dir, "s_vedai_b1_96x64.pt"))
    assert (g["config"], g["weight_seed"], g["input_seed"], g["fused"]) == ("yolov5s_fusion_transformerx3_vedai", 11, 12, False)
    z_ref, raw_ref = g["z"], g["raw"]
    cfg = cft.named_config(g["config"])
    sd = oracle.init_state(cfg, seed=11)
    x, x2 = oracle.make_inputs(1, 96, 64, seed=12)
    assert abs(float(x.double().sum()) - g["input_checksum"][0]) < 1e-6
    assert abs(float(x2.double().sum()) - g["input_checksum"][1]) < 1e-6
    assert abs(float(sum(v.double().abs().sum() for v in sd.values())) - g["state_checksum"]) < 1e-3
    z, raw = oracle.forward(sd, cfg, x, x2)
    assert_close_fp32(z[..., :4], z_ref[..., :4], 1e-5)
    assert_close_fp32(z[..., 4:], z_ref[..., 4:], 1e-5)
    for a, b in zip(raw, raw_ref):
        assert_close_fp32(a, b, 1e-6)
