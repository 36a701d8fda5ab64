"""CPU suite: checkpoint ingestion (SURVEY.md section 8f rank 3).  A checkpoint written exactly as the reference's
``train.py:850-857`` writes it (the UNMODIFIED reference ``Model``, ``.half()``, pickled whole) must load through
``attempt_load`` (mirror of ``models/experimental.py:113-134``) into a B200 ``Model`` with identical weights -- both with the
reference tree importable and, in a fresh interpreter WITHOUT it, through the ``models.*`` alias modules.  The checkpoint
is stored under tests/golden (written by oracle/make_golden.py)."""
import json
import lzma
import os
import shutil
import subprocess
import sys

import pytest
import torch

from oracle import ref_shim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = "yolov5s_fusion_transformerx3_vedai"


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory, golden_dir, cft, oracle):
    """The reference's ``Model`` of the s graph, seed-7 weights, pickled as train.py:850-857 writes it
    (oracle/make_golden.py), unpacked to a file.  The graph is the s graph at width multiple 1/64 instead of 0.5 (GPT
    d_model 8 / 8 / 16): the full-width checkpoint is about 90 MB, this one 179 KB compressed, and the loader walks the
    same 47 layers and state-dict keys either way."""
    cfg = dict(cft.named_config(NAME), width_multiple=1 / 64)
    sd = oracle.init_state(cfg, seed=7)
    path = str(tmp_path_factory.mktemp("ckpt") / "last.pt")
    with lzma.open(os.path.join(golden_dir, "ckpt_s_vedai_w64_half.pt.xz")) as src, open(path, "wb") as dst:
        shutil.copyfileobj(src, dst)
    return path, {k: v.half().float() if v.is_floating_point() else v for k, v in sd.items()}


def _summary(model):
    sd = model.state_dict()
    return {"layers": [type(m).__name__ for m in model.model], "modules": [type(m).__module__ for m in model.model],
            "n_keys": len(sd), "checksum": float(sum(v.double().abs().sum() for v in sd.values() if v.is_floating_point())),
            "names": model.names, "stride": [float(s) for s in model.stride], "save": list(model.save),
            "gpt_groups": {str(k): v for k, v in model._plan["gpt_groups"].items()}}


@pytest.mark.skipif(not ref_shim.available(), reason="needs the reference project's own Python modules")
def test_attempt_load_with_reference_importable(checkpoint, cft):
    """The checkpoint unpickles into the reference's own classes (no alias modules) and is converted from those."""
    from importlib import import_module
    path, sd_half = checkpoint
    ref_shim.import_reference()
    assert import_module(cft.__name__ + ".checkpoint")._reference_importable()
    model = cft.attempt_load(path, fuse=False)
    assert isinstance(model, cft.Model) and not model.training
    got = model.state_dict()
    assert set(got) == set(sd_half)
    for k, v in sd_half.items():
        assert torch.equal(got[k].float(), v.float()), k
    assert all(type(m).__module__.startswith("multispectral-object-detection_b200") or type(m).__name__ == "Upsample"
               for m in model.model)
    assert model._plan["gpt_groups"] and model.names[0] == "cls0"
    fused = cft.attempt_load(path)                                         # default: .fuse() like the reference
    assert not any(hasattr(m, "bn") for m in fused.modules() if type(m).__name__ == "Conv")


def test_attempt_load_without_the_reference_tree(checkpoint, cft):
    path, _ = checkpoint
    ref = _summary(cft.attempt_load(path, fuse=False))
    code = (
        "import sys, json, importlib\n"
        f"sys.path = [p for p in sys.path if 'reference' not in p]; sys.path.insert(0, {ROOT!r})\n"
        "assert 'models' not in sys.modules\n"
        "cft = importlib.import_module('multispectral-object-detection_b200')\n"
        "sys.path.insert(0, %r)\n" % os.path.join(ROOT, "tests") +
        "from test_checkpoint_cpu import _summary\n"
        f"m = cft.attempt_load({path!r}, fuse=False)\n"
        "assert 'models' not in sys.modules, 'alias modules must not leak'\n"
        "print('SUMMARY ' + json.dumps(_summary(m)))\n")
    env = {k: v for k, v in os.environ.items() if k not in ("PYTHONPATH", "CFT_REFERENCE_ROOT")}
    env["CFT_REFERENCE_ROOT"] = "/nonexistent"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600, cwd="/tmp")
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("SUMMARY ")][-1]
    got = json.loads(line[len("SUMMARY "):])
    assert got == json.loads(json.dumps(ref))


def test_attempt_load_rejects_ensembles(cft):
    with pytest.raises(cft.CftError):
        cft.attempt_load(["a.pt", "b.pt"])
