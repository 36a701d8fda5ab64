"""The drop-in boundary exercised ON THE GPU with the UNMODIFIED reference's own code (SURVEY.md section 8b; VERDICT r1
items 4-6).  The tests that drive the reference's own modules need its tree (``oracle/ref_shim.py``) and skip without it;
the comparison with the reference's forward reads its stored outputs (``tests/golden``, oracle/make_golden.py).

* ``install()``: the reference's ``parse_model`` (``models/yolo_test.py:479-555``, ``eval`` of the yaml names at ``:488``)
  builds the B200 classes, and the reference's ``Model.forward`` / ``forward_once`` (``:214-272``) -- its own layer walk,
  its own ``y`` / ``save`` bookkeeping, no planner -- drives the CUDA kernels; result vs the fp32 CPU oracle.
* ``convert()``: a model built from the reference's PyTorch modules is swapped module by module, keeps its weights.
* ``attempt_load()``: a checkpoint pickled by the reference exactly as ``train.py:850-857`` writes it (``.half()``, whole
  model) loads into a B200 ``Model`` and forwards on the GPU; vs the oracle on the fp16-rounded weights.
Tolerances: those of tests/test_model_gpu.py (``check_outputs``)."""
import os

import pytest
import torch

from oracle import ref_shim
from parity_util import anchor_grid_of, check_outputs

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not ref_shim.available(), reason="needs the reference project's own Python modules")
DEV = "cuda"
NAME = "yolov5s_fusion_transformerx3_vedai"


@pytest.fixture(scope="module")
def yt():
    return ref_shim.import_reference()


@needs_reference
def test_reference_model_and_forward_once_run_on_the_b200_kernels(yt, cft, oracle):
    cfg = cft.named_config(NAME)
    sd = oracle.init_state(cfg, seed=11)
    prev = cft.install(yt)
    try:
        rm = yt.Model(ref_shim.reference_yaml(NAME), ch=3)          # the reference's own Model.__init__ / parse_model
    finally:
        cft.uninstall(yt, prev)
    assert type(rm).__module__ == "models.yolo_test"
    assert {type(m).__module__ for m in rm.model} == {"multispectral-object-detection_b200.modules"}
    rm.load_state_dict(sd, strict=True)
    rm = rm.to(DEV).eval()
    x, x2 = oracle.make_inputs(2, 128, 160, seed=12)
    n0 = cft._lib.launch_count()
    with torch.no_grad():
        z, raw = rm(x.to(DEV), x2.to(DEV))                          # reference Model.forward -> forward_once (:214-272)
    torch.cuda.synchronize()
    assert cft._lib.launch_count() - n0 > 60                        # the library's kernels ran, not PyTorch ops
    z_ref, raw_ref = oracle.forward(sd, cfg, x, x2)
    print(check_outputs(z, raw, z_ref, raw_ref, oracle, anchor_grid_of(sd)))
    # the same weights through the stand-alone mirror (planner, fused Add2/Add): same function
    mirror = cft.Model(cfg).eval()
    mirror.load_state_dict(sd, strict=True)
    with torch.no_grad():
        z_m, raw_m = mirror.to(DEV)(x.to(DEV), x2.to(DEV))
    torch.cuda.synchronize()
    for a, b in zip(raw, raw_m):
        assert float((a.float() - b.float()).norm() / b.float().norm()) <= 1e-2


@needs_reference
def test_reference_fuse_then_forward(yt, cft, oracle):
    """Model.fuse() of the reference (models/yolo_test.py:296-304: `type(m) is Conv and hasattr(m, 'bn')`) on the installed classes."""
    cfg = cft.named_config(NAME)
    sd = oracle.init_state(cfg, seed=13)
    prev = cft.install(yt)
    try:
        rm = yt.Model(ref_shim.reference_yaml(NAME), ch=3)
        rm.load_state_dict(sd, strict=True)
        rm = rm.eval().fuse()                                      # needs the rebound `Conv` global: inside install()
    finally:
        cft.uninstall(yt, prev)
    assert not any(hasattr(m, "bn") for m in rm.modules() if type(m).__name__ == "Conv")
    rm = rm.to(DEV)
    x, x2 = oracle.make_inputs(1, 96, 96, seed=14)
    with torch.no_grad():
        z, raw = rm(x.to(DEV), x2.to(DEV))
    torch.cuda.synchronize()
    z_ref, raw_ref = oracle.forward(sd, cfg, x, x2)
    print(check_outputs(z, raw, z_ref, raw_ref, oracle, anchor_grid_of(sd)))


@needs_reference
def test_convert_reference_pytorch_model(yt, cft, oracle):
    cfg = cft.named_config(NAME)
    sd = oracle.init_state(cfg, seed=15)
    rm = yt.Model(ref_shim.reference_yaml(NAME), ch=3)
    assert type(rm.model[0]).__module__ == "models.common"          # the reference's PyTorch modules
    rm.load_state_dict(sd, strict=True)
    rm = cft.convert(rm.eval()).to(DEV)
    x, x2 = oracle.make_inputs(1, 128, 96, seed=16)
    with torch.no_grad():
        z, raw = rm(x.to(DEV), x2.to(DEV))
    torch.cuda.synchronize()
    z_ref, raw_ref = oracle.forward(sd, cfg, x, x2)
    print(check_outputs(z, raw, z_ref, raw_ref, oracle, anchor_grid_of(sd)))


@needs_reference
def test_attempt_load_checkpoint_forward(yt, cft, oracle, tmp_path):
    from copy import deepcopy
    cfg = cft.named_config(NAME)
    sd = oracle.init_state(cfg, seed=17)
    rm = yt.Model(ref_shim.reference_yaml(NAME), ch=3)
    rm.load_state_dict(sd, strict=True)
    rm.names = [f"cls{i}" for i in range(cfg["nc"])]
    path = str(tmp_path / "last.pt")
    torch.save({"epoch": 1, "best_fitness": 0.1, "training_results": "", "model": deepcopy(rm).half(), "ema": None,
                "updates": 0, "optimizer": None, "wandb_id": None}, path)          # train.py:850-857
    model = cft.attempt_load(path, map_location="cpu").to(DEV)      # models/experimental.py:113-134: .float().fuse().eval()
    assert isinstance(model, cft.Model) and not model.training
    x, x2 = oracle.make_inputs(1, 128, 128, seed=18)
    with torch.no_grad():
        z, raw = model(x.to(DEV), x2.to(DEV))
    torch.cuda.synchronize()
    sd_half = {k: (v.half().float() if v.is_floating_point() else v) for k, v in sd.items()}
    z_ref, raw_ref = oracle.forward(sd_half, cfg, x, x2)
    print(check_outputs(z, raw, z_ref, raw_ref, oracle, anchor_grid_of(sd_half)))


def test_reference_pytorch_modules_on_gpu_vs_ours(cft, oracle, golden_dir):
    """The reference's own modules (fp32 eager forward, stored by oracle/make_golden.py) and the B200 kernels agree: the
    eager-GPU baseline of bench.py is a forward of the same function."""
    g = torch.load(os.path.join(golden_dir, "s_vedai_b1_128x128.pt"))
    assert (g["config"], g["weight_seed"], g["input_seed"], g["fused"]) == (NAME, 19, 20, False)
    cfg = cft.named_config(NAME)
    sd = oracle.init_state(cfg, seed=19)
    ours = cft.Model(cfg).eval()
    ours.load_state_dict(sd, strict=True)
    ours = ours.to(DEV)
    x, x2 = oracle.make_inputs(1, 128, 128, seed=20)
    assert abs(float(x.double().sum()) - g["input_checksum"][0]) < 1e-6
    assert abs(float(x2.double().sum()) - g["input_checksum"][1]) < 1e-6
    with torch.no_grad():
        z_o, raw_o = ours(x.to(DEV), x2.to(DEV))
    torch.cuda.synchronize()
    print(check_outputs(z_o, raw_o, g["z"], g["raw"], oracle, anchor_grid_of(sd)))
