"""Generate tests/golden/nms_cases.pt and nms_seed21_cases.pt from the UNMODIFIED reference
``utils.general.non_max_suppression`` (build container only; TEST INFRASTRUCTURE).

For each seeded case (``nms_oracle.make_predictions``) run the reference function (which calls the installed
torchvision.ops.nms), assert the CPU restatement ``nms_oracle.non_max_suppression`` reproduces it bit for bit, and
store the REFERENCE's outputs plus a float64 checksum of the inputs, so the GPU box (no ``/root/reference``) can
check that it regenerated the same inputs.

    python oracle/make_golden_nms.py
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import nms_oracle as N  # noqa: E402
from oracle import ref_shim  # noqa: E402

# name, (b, rows, nc, seed), make_predictions kwargs, non_max_suppression kwargs
CASES = [
    ("default_b2_3000_nc3", (2, 3000, 3, 0), {}, {}),
    ("multilabel_b1_8000_nc9", (1, 8000, 9, 1), {}, {"multi_label": True}),
    ("multilabel_nc1_is_off", (2, 2500, 1, 2), {}, {"multi_label": True}),
    ("agnostic_b2_3000_nc3", (2, 3000, 3, 3), {}, {"agnostic": True}),
    ("classes_1_3_of_5", (2, 3000, 5, 4), {}, {"classes": [1, 3]}),
    ("full_640_lowconf", (1, 25200, 3, 5), {}, {"conf_thres": 0.001, "iou_thres": 0.6}),
    ("over_max_nms_multilabel", (1, 12000, 3, 6), {}, {"multi_label": True, "conf_thres": 0.001, "iou_thres": 0.6}),
    ("nothing_passes", (2, 500, 3, 7), {}, {"conf_thres": 0.99}),
    ("few_boxes_b3_40_nc2", (3, 40, 2, 8), {"clusters": 3}, {}),
    ("sparse_scene", (2, 6000, 3, 9), {"clusters": 400, "conf_lo": 0.2}, {"iou_thres": 0.3}),
]

# one seeded batch under each branch of the keyword arguments (tests/test_nms_cpu.py)
SEED21_CASES = [
    ("seed21_default", (2, 2000, 3, 21), {}, {}),
    ("seed21_multilabel", (2, 2000, 3, 21), {}, {"multi_label": True}),
    ("seed21_agnostic_iou03", (2, 2000, 3, 21), {}, {"agnostic": True, "iou_thres": 0.3}),
    ("seed21_classes_0", (2, 2000, 3, 21), {}, {"classes": [0]}),
]


def main():
    ref_shim.import_reference()
    for file, cases in (("nms_cases.pt", CASES), ("nms_seed21_cases.pt", SEED21_CASES)):
        write(cases, os.path.join(ROOT, "tests", "golden", file))


def write(cases, path):
    from utils.general import non_max_suppression as ref_nms  # the reference's own function
    golden = {}
    for name, (b, rows, nc, seed), pk, kw in cases:
        p = N.make_predictions(b, rows, nc, seed, **pk)
        ref = ref_nms(p.clone(), **kw)
        mine = N.non_max_suppression(p, **kw)
        assert len(ref) == len(mine)
        for r, m in zip(ref, mine):
            assert r.shape == m.shape and torch.equal(r, m), f"{name}: oracle != reference"
        golden[name] = {"args": (b, rows, nc, seed), "pred_kwargs": pk, "nms_kwargs": kw,
                        "input_checksum": float(p.double().sum()), "out": [r.clone() for r in ref]}
        print(f"{name}: {[tuple(r.shape) for r in ref]} oracle == reference")
    torch.save(golden, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
