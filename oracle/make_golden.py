"""Generate tests/golden/*.pt from the UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE.  For each case: build the reference ``models.yolo_test.Model`` from the
reference's own yaml (or, for the derived yolov5x x3 graph, from the dict), load the seeded
synthetic state (``cft_oracle.init_state``), run the reference eval forward on CPU fp32,
assert the CPU restatement (``cft_oracle.forward``) reproduces it, and store the REFERENCE's
outputs plus float64 checksums of the seeded inputs/weights so the GPU box (which has no
``/root/reference``) can verify it regenerated the same tensors.

It also stores the other things the tests compare against the reference: ``yaml.safe_load`` of the reference's x3 graph
files (``reference_x3_yaml.json``) and a checkpoint pickled by the reference's own ``Model`` exactly as its ``train.py``
writes one, of a width-1/64 variant of the s graph, xz-compressed so that it stays small (``ckpt_s_vedai_w64_half.pt.xz``).

    python oracle/make_golden.py [name ...]    # writes only the named goldens (a case, reference_x3_yaml or
                                               # ckpt_s_vedai_w64_half); without names, every case and both files
"""
import importlib
import json
import lzma
import os
import sys
from copy import deepcopy

import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import cft_oracle as O  # noqa: E402
from oracle import ref_shim  # noqa: E402

config = importlib.import_module("multispectral-object-detection_b200.config")

# name, config-name, batch, H, W, weight seed, input seed, fused
CASES = [
    ("s_vedai_b2_128x160", "yolov5s_fusion_transformerx3_vedai", 2, 128, 160, 0, 1, False),
    ("s_vedai_b1_64x64_fused", "yolov5s_fusion_transformerx3_vedai", 1, 64, 64, 3, 4, True),
    ("l_flir_b1_64x64", "yolov5l_fusion_transformerx3_FLIR_aligned", 1, 64, 64, 0, 1, False),
    ("l_llvip_b1_64x96", "yolov5l_fusion_transformerx3_llvip", 1, 64, 96, 5, 6, False),
    ("x_flir_b1_64x64", "yolov5x_fusion_transformerx3_FLIR_aligned", 1, 64, 64, 0, 1, False),
    ("s_vedai_b1_96x64", "yolov5s_fusion_transformerx3_vedai", 1, 96, 64, 11, 12, False),
    ("s_vedai_b1_128x128", "yolov5s_fusion_transformerx3_vedai", 1, 128, 128, 19, 20, False),
]

YAML_NAMES = ["yolov5l_fusion_transformerx3_FLIR_aligned", "yolov5l_fusion_transformerx3_llvip",
              "yolov5s_fusion_transformerx3_vedai"]

# the checkpoint: the s graph at width 1/64 (GPT d_model 8 / 8 / 16), weight seed 7
CKPT_NAME, CKPT_WIDTH, CKPT_SEED = "yolov5s_fusion_transformerx3_vedai", 1 / 64, 7


def checkpoint_config():
    return dict(config.named_config(CKPT_NAME), width_multiple=CKPT_WIDTH)


def checksum(t):
    return float(t.double().sum())


def state_checksum(sd):
    return float(sum(v.double().abs().sum() for v in sd.values()))


def write_yaml_configs(out_dir):
    configs = {}
    for name in YAML_NAMES:
        with open(ref_shim.reference_yaml(name)) as f:
            configs[name] = yaml.safe_load(f)
    with open(os.path.join(out_dir, "reference_x3_yaml.json"), "w") as f:
        json.dump(configs, f, indent=1)
        f.write("\n")


def write_checkpoint(yt, out_dir):
    cfg = checkpoint_config()
    model = yt.Model(cfg, ch=3)
    model.load_state_dict(O.init_state(cfg, seed=CKPT_SEED), strict=True)
    model.names = [f"cls{i}" for i in range(cfg["nc"])]
    ckpt = {"epoch": 3, "best_fitness": 0.5, "training_results": "", "model": deepcopy(model).half(), "ema": None,
            "updates": 0, "optimizer": None, "wandb_id": None}                       # train.py:850-857
    path = os.path.join(out_dir, "ckpt_s_vedai_w64_half.pt.xz")
    with lzma.open(path, "wb", preset=9) as f:
        torch.save(ckpt, f)
    print(f"{path}: {os.path.getsize(path)} bytes")


def main(names):
    yt = ref_shim.import_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    if not names or "reference_x3_yaml" in names:
        write_yaml_configs(out_dir)
    if not names or "ckpt_s_vedai_w64_half" in names:
        write_checkpoint(yt, out_dir)
    for name, cname, b, h, w, wseed, iseed, fused in CASES:
        if names and name not in names:
            continue
        cfg = config.named_config(cname)
        ypath = ref_shim.reference_yaml(cname)
        model = yt.Model(ypath if os.path.isfile(ypath) else cfg, ch=3).eval()
        sd = O.init_state(cfg, seed=wseed)
        model.load_state_dict(sd, strict=True)
        if fused:
            model.fuse()                      # models/yolo_test.py:296-304
        x, x2 = O.make_inputs(b, h, w, seed=iseed)
        with torch.no_grad():
            z_ref, raw_ref = model(x, x2)
        osd = {k: v for k, v in model.state_dict().items()} if fused else sd
        z_o, raw_o = O.forward(osd, cfg, x, x2)
        dz = (z_ref - z_o).abs().max().item()
        dr = max((a - c).abs().max().item() for a, c in zip(raw_ref, raw_o))
        assert dz <= 1e-4 and dr <= 1e-5, (name, dz, dr)
        torch.save({
            "case": name, "config": cname, "batch": b, "height": h, "width": w,
            "weight_seed": wseed, "input_seed": iseed, "fused": fused,
            "z": z_ref.clone(), "raw": [r.clone() for r in raw_ref],
            "input_checksum": [checksum(x), checksum(x2)],
            "state_checksum": state_checksum(sd),
            "oracle_vs_reference_max_abs": [dz, dr],
            "torch": str(torch.__version__),
        }, os.path.join(out_dir, name + ".pt"))
        print(f"{name}: z{tuple(z_ref.shape)} oracle-vs-reference max|d| z={dz:.2e} raw={dr:.2e}")


if __name__ == "__main__":
    main(sys.argv[1:])
