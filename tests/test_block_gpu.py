"""GPU parity tests of the one-launch transformer stack (``cft_gpt_block``, csrc/cft_block.cu) against
(a) a plain fp32 PyTorch restatement of models/common.py:475-513,540-546,622-625 on the same (bf16-rounded) weights and
(b) the per-op path of the same library (LN / GEMM / attention launches), which rounds at the same places.

Tolerances: vs fp32 torch, rel-L2 <= 1e-2 and max|d| <= 6e-2 * max|ref| on the ln_f output (bf16 GEMM operands: LN outputs,
q/k/v, P, O and the MLP hidden are rounded to bf16, 8 layers deep); vs the per-op path max|d| <= 2e-2 * max|ref|
(identical rounding points; the one-pass variance and the fp32 summation order differ)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"


def make_gpt(cft, d, layers, seed):
    torch.manual_seed(seed)
    g = cft.modules.GPT(d, n_layer=layers).eval()
    with torch.no_grad():
        for m in g.modules():
            if isinstance(m, torch.nn.Linear):
                m.weight.normal_(0.0, 1.0 / math.sqrt(m.in_features))
                m.bias.normal_(0.0, 0.1)
                m.weight.copy_(m.weight.to(torch.bfloat16).float())       # both sides see the same weights
            elif isinstance(m, torch.nn.LayerNorm):
                m.weight.uniform_(0.5, 1.5)
                m.bias.normal_(0.0, 0.1)
    return g.to(DEV)


def ref_stack(g, x, upto=None):
    """fp32 restatement; returns (ln_f output, [x after every layer])."""
    h = g.h
    xs = []
    for blk in list(g.trans_blocks)[:upto]:
        b, t, c = x.shape
        y = F.layer_norm(x, (c,), blk.ln_input.weight, blk.ln_input.bias, blk.ln_input.eps)
        sa = blk.sa
        q = sa.que_proj(y).view(b, t, h, c // h).permute(0, 2, 1, 3)
        k = sa.key_proj(y).view(b, t, h, c // h).permute(0, 2, 3, 1)
        v = sa.val_proj(y).view(b, t, h, c // h).permute(0, 2, 1, 3)
        att = torch.softmax(q @ k / math.sqrt(c // h), -1)
        o = (att @ v).permute(0, 2, 1, 3).reshape(b, t, c)
        x = x + sa.out_proj(o)
        y = F.layer_norm(x, (c,), blk.ln_output.weight, blk.ln_output.bias, blk.ln_output.eps)
        x = x + blk.mlp[2](F.gelu(blk.mlp[0](y)))
        xs.append(x)
    return F.layer_norm(x, (x.shape[-1],), g.ln_f.weight, g.ln_f.bias, g.ln_f.eps), xs


CASES = [
    # d, layers, B, cluster (0 = auto)
    (256, 8, 3, 0),       # yolov5l P3: cluster 4, DC 64, dk 32 (SWIZZLE_64B q/k/v tiles), 2 heads per CTA
    (512, 8, 2, 0),       # yolov5l P4 / yolov5s P5: cluster 4, DC 128, dk 64 (P aliases Q|K), 16 KiB weight stages
    (512, 2, 3, 4),       # the same split forced
    (128, 8, 2, 0),       # yolov5s P3: cluster 2, dk 16 (SWIZZLE_32B tiles), 4 heads per CTA = two head pairs
    (256, 1, 45, 4),      # more images than co-resident clusters: clusters loop over images
    (256, 8, 3, 2),       # the d = 256 plan of batches 34-66: cluster 2, DC 128, dk 32, 4 heads per CTA = two head pairs
]


@pytest.mark.parametrize("d,layers,B,cluster", CASES)
def test_gpt_block_vs_fp32_and_per_op(d, layers, B, cluster, cft):
    g = make_gpt(cft, d, layers, seed=d + layers)
    gen = torch.Generator().manual_seed(7)
    tok = (torch.randn(B, 128, d, generator=gen) * 0.7 + 0.1).to(DEV)
    w = g._weights(torch.device(DEV))
    assert cft.ops.gpt_block_supported(B, d, g.h, 128)
    dbg = torch.zeros(layers, B, 128, d, device=DEV)
    out = cft.ops.gpt_block(tok, w["stack"], g.h, cluster=cluster, debug_x=dbg)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref, xs = ref_stack(g, tok)
    for l, xr in enumerate(xs):                      # per-layer residual stream: localises a failure
        rel = float((dbg[l] - xr).norm() / xr.norm())
        assert rel <= 1.5e-2, f"x after layer {l}: rel-L2 {rel:.4f}"
    rel = float((out - ref).norm() / ref.norm())
    mx = float((out - ref).abs().max() / ref.abs().max())
    assert rel <= 1e-2 and mx <= 6e-2, f"ln_f output: rel-L2 {rel:.4f} max {mx:.4f}"
    # the per-op path of the same library
    x2d = tok.view(B * 128, d).clone()
    ops = cft.ops
    for L in w["layers"]:
        y = ops.layernorm(x2d, *L["ln1"])
        qkv = ops.gemm(y, L["qkv"][0], L["qkv"][1])
        att = ops.attention(qkv, B, 128, d, g.h)
        x2d = ops.gemm(att, L["out"][0], L["out"][1], residual=x2d, out_dtype=torch.float32)
        y = ops.layernorm(x2d, *L["ln2"])
        hid = ops.gemm(y, L["up"][0], L["up"][1], act=ops.ACT_GELU)
        x2d = ops.gemm(hid, L["down"][0], L["down"][1], residual=x2d, out_dtype=torch.float32)
    per_op = ops.layernorm(x2d, *w["lnf"], out_dtype=torch.float32).view(B, 128, d)
    torch.cuda.synchronize()
    mx2 = float((out - per_op).abs().max() / per_op.abs().max())
    assert mx2 <= 2e-2, f"fused vs per-op path: max {mx2:.4f}"


def test_gpt_block_batch_invariant_and_deterministic(cft):
    """An image's result must not depend on the batch it is in or on which cluster ran it (bit-exact)."""
    d, B = 256, 9
    g = make_gpt(cft, d, 8, seed=3)
    tok = (torch.randn(B, 128, d, generator=torch.Generator().manual_seed(5)) * 0.5).to(DEV)
    w = g._weights(torch.device(DEV))["stack"]
    a = cft.ops.gpt_block(tok, w, g.h)
    b = cft.ops.gpt_block(tok, w, g.h)
    one = cft.ops.gpt_block(tok[4:5].contiguous(), w, g.h)
    perm = torch.arange(B - 1, -1, -1, device=DEV)
    c = cft.ops.gpt_block(tok[perm].contiguous(), w, g.h)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert torch.equal(a[4:5], one)
    assert torch.equal(a[perm], c)


def test_gpt_tokens_module_uses_fused_block(cft):
    """GPT.tokens through the module (tokeniser + fused stack) equals the per-op path within the bf16 bound, and takes
    3 launches instead of 58."""
    d, B = 256, 2
    g = make_gpt(cft, d, 8, seed=11)
    rgb = torch.randn(B, d, 20, 20, generator=torch.Generator().manual_seed(1)).to(DEV).to(torch.bfloat16)
    ir = torch.randn(B, d, 20, 20, generator=torch.Generator().manual_seed(2)).to(DEV).to(torch.bfloat16)
    rgb, ir = (t.contiguous(memory_format=torch.channels_last) for t in (rgb, ir))
    n0 = cft._lib.launch_count()
    fused = g.tokens(rgb, ir)
    n1 = cft._lib.launch_count()
    g.fused_block = False
    try:
        per_op = g.tokens(rgb, ir)
    finally:
        del g.fused_block
    n2 = cft._lib.launch_count()
    torch.cuda.synchronize()
    assert n1 - n0 == 2 and n2 - n1 == 2 + 7 * 8, (n1 - n0, n2 - n1)
    assert float((fused - per_op).abs().max() / per_op.abs().max()) <= 2e-2
