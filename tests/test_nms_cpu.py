"""CPU suite for the NMS row (SURVEY.md §8f rank 2): the CPU restatement ``oracle/nms_oracle.py`` against the committed
golden outputs of the UNMODIFIED reference ``utils.general.non_max_suppression`` (oracle/make_golden_nms.py).
Bit-exact."""
import os

import pytest
import torch

from oracle import nms_oracle as N


def _golden(golden_dir):
    return torch.load(os.path.join(golden_dir, "nms_cases.pt"))


def test_nms_golden_covers_every_branch(golden_dir):
    g = _golden(golden_dir)
    kws = [c["nms_kwargs"] for c in g.values()]
    assert any(k.get("multi_label") for k in kws) and any(k.get("agnostic") for k in kws)
    assert any(k.get("classes") for k in kws)
    assert any(sum(o.shape[0] for o in c["out"]) == 0 for c in g.values())                 # nothing passes
    assert any(c["args"][1] * (c["args"][2] if c["nms_kwargs"].get("multi_label") else 1) > N.MAX_NMS
               for c in g.values())                                                         # > max_nms candidates
    assert any(any(o.shape[0] == N.MAX_DET for o in c["out"]) for c in g.values())         # max_det cap hit


def test_nms_oracle_matches_reference_golden(golden_dir):
    for name, c in _golden(golden_dir).items():
        b, rows, nc, seed = c["args"]
        p = N.make_predictions(b, rows, nc, seed, **c["pred_kwargs"])
        assert abs(float(p.double().sum()) - c["input_checksum"]) < 1e-6, name     # same inputs as the reference saw
        out = N.non_max_suppression(p, **c["nms_kwargs"])
        assert len(out) == len(c["out"])
        for a, r in zip(out, c["out"]):
            assert a.shape == r.shape and torch.equal(a, r), name


def test_nms_oracle_properties():
    p = N.make_predictions(2, 4000, 4, seed=11)
    out = N.non_max_suppression(p, conf_thres=0.3, iou_thres=0.5)
    for d in out:
        assert d.shape[0] <= N.MAX_DET and (d[:, 4] > 0.3).all()
        assert (d[1:, 4] <= d[:-1, 4]).all()                                        # descending confidence
        # no kept pair of one class overlaps by more than the threshold
        import torchvision
        iou = torchvision.ops.box_iou(d[:, :4], d[:, :4])
        same = d[:, 5:6] == d[:, 5:6].T
        iou = iou * same - torch.eye(d.shape[0])
        assert iou.max() <= 0.5 + 1e-6


@pytest.mark.parametrize("kw", [{}, {"multi_label": True}, {"agnostic": True, "iou_thres": 0.3}, {"classes": [0]}])
def test_nms_oracle_equals_stored_reference(kw, golden_dir):
    """One seeded batch under each branch of the keyword arguments, against the reference function's stored outputs."""
    case = [c for c in torch.load(os.path.join(golden_dir, "nms_seed21_cases.pt")).values() if c["nms_kwargs"] == kw]
    assert len(case) == 1 and case[0]["args"] == (2, 2000, 3, 21)
    p = N.make_predictions(2, 2000, 3, seed=21)
    assert abs(float(p.double().sum()) - case[0]["input_checksum"]) < 1e-6        # same inputs as the reference saw
    ref = case[0]["out"]
    out = N.non_max_suppression(p, **kw)
    assert len(out) == len(ref)
    for a, r in zip(out, ref):
        assert a.shape == r.shape and torch.equal(a, r)


def test_nms_wrapper_fails_loudly_without_cuda(cft):
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from importlib import import_module
    nms = import_module("multispectral-object-detection_b200.nms")
    with pytest.raises(cft.CftError):
        nms.non_max_suppression(torch.rand(1, 10, 8))


# ---------------------------------------------------------------------------------------------------------------------
# The two algorithmic claims csrc/nms.cu rests on, emulated step by step in Python (the kernel itself is covered by
# tests/test_nms_gpu.py): (1) the all-ascending bitonic network with VIRTUAL +inf padding sorts any n, (2) resolving
# the sorted candidates in chunks, one 32-candidate batch per round (kept-list test -> 32x32 suppression matrix ->
# serial scan over its rows -> broadcast of the newly kept boxes), is the sequential greedy suppression.
# ---------------------------------------------------------------------------------------------------------------------
def _bitonic_virtual_padding(keys):
    import numpy as np
    k_ = np.array(keys, dtype=np.uint64)
    n = len(k_)
    n2 = 1
    while n2 < n:
        n2 <<= 1

    def step(pair_of):
        for t in range(n2 >> 1):
            i, l = pair_of(t)
            if l < n and k_[i] > k_[l]:                     # pairs whose upper index is padding are skipped
                k_[i], k_[l] = k_[l], k_[i]
    k, lk = 2, 1
    while k <= n2:
        hk = k >> 1
        step(lambda t: (((t >> (lk - 1)) << lk) + (t & (hk - 1)), ((t >> (lk - 1)) << lk) + k - 1 - (t & (hk - 1))))
        j = hk >> 1
        while j >= 1:
            step(lambda t, j=j: (((t & ~(j - 1)) << 1) | (t & (j - 1)), (((t & ~(j - 1)) << 1) | (t & (j - 1))) + j))
            j >>= 1
        k <<= 1
        lk += 1
    return k_


def test_kernel_sort_network_with_virtual_padding():
    import numpy as np
    rng = np.random.default_rng(0)
    for n in (0, 1, 2, 3, 5, 17, 100, 257, 1000, 1025, 1500):
        a = rng.integers(0, 40, size=n).astype(np.uint64)       # many ties
        assert (_bitonic_virtual_padding(a) == np.sort(a)).all(), n


def _chunked_greedy(boxes, scores, thr, max_det, chunk=64, warp=8):
    """csrc/nms.cu phase 3 with `chunk` threads of `warp` lanes (the kernel: 1024 / 32)."""
    import numpy as np
    f = np.float32
    thr = f(thr)

    def gt(a, b):                                              # iou_gt(a = earlier box, b = later box)
        w = max(f(0), f(min(a[2], b[2]) - max(a[0], b[0])))
        h = max(f(0), f(min(a[3], b[3]) - max(a[1], b[1])))
        inter = f(w * h)
        if inter == 0 and thr >= 0:
            return False
        with np.errstate(all="ignore"):
            return f(inter / f(f(a[4] + b[4]) - inter)) > thr
    n = len(scores)
    order = np.argsort(-scores, kind="stable")
    area = ((boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1])).astype(f)
    cand = [(boxes[i, 0], boxes[i, 1], boxes[i, 2], boxes[i, 3], area[i]) for i in order]
    kept, kept_idx = [], []
    for base in range(0, n, chunk):
        if len(kept) >= max_det:
            break
        m = min(chunk, n - base)
        alive = [t < m and not any(gt(kb, cand[base + t]) for kb in kept) for t in range(chunk)]
        while True:
            kept_before = len(kept)
            if kept_before >= max_det:
                break
            warps_alive = [any(alive[w * warp:(w + 1) * warp]) for w in range(chunk // warp)]
            if not any(warps_alive):
                break
            fw = warps_alive.index(True)
            lanes = list(range(fw * warp, (fw + 1) * warp))
            sup = {l: {l2 for l2 in lanes if l2 > l and l2 < m and l < m and gt(cand[base + l], cand[base + l2])} for l in lanes}
            remaining = [l for l in lanes if alive[l]]
            room = max_det - kept_before
            while remaining and room > 0:
                l = remaining.pop(0)
                kept.append(cand[base + l])
                kept_idx.append(int(order[base + l]))
                room -= 1
                remaining = [x for x in remaining if x not in sup[l]]
            for l in lanes:
                alive[l] = False
            for t in range(m):
                if alive[t] and any(gt(kb, cand[base + t]) for kb in kept[kept_before:]):
                    alive[t] = False
    return kept_idx


@pytest.mark.parametrize("seed,max_det", [(0, 300), (1, 20), (2, 300), (3, 7)])
def test_kernel_round_structure_equals_sequential_greedy(seed, max_det):
    p = N.make_predictions(1, 600, 3, seed)[0].numpy()
    box, sc = N.xywh2xyxy(p[:, :4]), p[:, 4]
    ref = N.nms_greedy(box, sc, 0.45, limit=max_det).tolist()
    assert _chunked_greedy(box, sc, 0.45, max_det) == ref


@pytest.mark.parametrize("seed", range(12))
def test_nms_greedy_equals_installed_torchvision(seed):
    """``nms_greedy`` (the restated CPU algorithm) against the installed ``torchvision.ops.nms`` itself, on random boxes,
    thresholds and heavy score ties -- kept indices identical and in the same order."""
    import numpy as np
    import torchvision
    g = torch.Generator().manual_seed(1000 + seed)
    n = int(torch.randint(1, 1500, (1,), generator=g))
    xy = torch.rand(n, 2, generator=g) * 200
    wh = torch.rand(n, 2, generator=g) * 80 + 1
    boxes = torch.cat([xy, xy + wh], 1)
    scores = torch.rand(n, generator=g)
    if seed % 3 == 0:
        scores = (scores * 8).floor() / 8                       # only 8 distinct scores: the stable order decides
    if seed % 4 == 1:
        boxes[n // 2:] = boxes[: n - n // 2].clone()            # exact duplicates
    thr = float(torch.rand(1, generator=g)) * 0.9
    ref = torchvision.ops.nms(boxes, scores, thr).numpy()
    mine = N.nms_greedy(boxes.numpy(), scores.numpy(), thr)
    assert mine.shape == ref.shape and (mine == ref).all()
