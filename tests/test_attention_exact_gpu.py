"""GPU tests of the attention core and the one-launch transformer stack whose expected answer is known exactly:

1. Per-op attention (``cft_attention``: the tcgen05 kernel, and the CUDA-core kernel for T < 128, for head dims the
   tensor-core split does not cover and under CFT_ATTENTION_SIMT=1).  q / k are c * (+-1 codes): key s of a head carries
   the code of an index, the query t the code of its target, so the scores peak at the target with a gap of >= 2 c^2 --
   large enough that every other key's exp2 is 0 in fp32 -- and the peak's P is exactly 1.  v holds integers in
   [-16, 16], so out[t] = v[target(t)] bit for bit.  Keys may share a code (groups of 2 .. 64 keys, and q = 0 for uniform
   attention over all 128): out = bf16_rn(exact group mean).  Every index bit of a code lives in one head-dim chunk of the
   tcgen05 split only, so a chunk that is dropped or mis-addressed ties keys and changes the output; bit 0 fills the first
   8 columns, so reading the next head's 8 columns where the last chunk overhangs dk (dk = 8 mod 16) ties or flips keys
   too (checked on the host for every case).  Large logits (max |S| ~ 1e7): P of the peak is no longer 1, the output
   p v / p must still be v exactly.
2. The fused stack (``cft_gpt_block`` with ``debug_x``) and the per-op path, every layer bit for bit.  Token rows are
   balanced +-1 (mean 0, variance 1, so LayerNorm gives +-gamma + beta exactly in bf16); one of three layers is nonzero:
   hard attention (Wk / Wq select code blocks of the row, Wv sparse +-1, Wo a signed permutation), uniform attention
   (Wq = 0), or an MLP whose pre-activations are >= 24 or <= -24 (GELU returns v or -0 exactly).  A zero layer adds
   exactly 0, so x after every layer is known exactly: a weight row read from the wrong layer, a key of the wrong image or
   head, or a hidden slice at the wrong K offset fails bit for bit.  Every fused plan for heads = 8 runs, plus clusters
   that loop over images.

Every case asserts on the host that its operands meet the exactness conditions: bf16-exact integers, partial sums below
2^24, the score gap, and max |S| below the limit where the kernel's P of the peak stops rounding to 1."""
import math
import os

import numpy as np
import pytest
import torch

from test_block_gpu import make_gpt
from test_exact_gpu import _ln_check

pytestmark = pytest.mark.gpu
DEV = "cuda"
T = 128
LOG2E = math.log2(math.e)
SIMT = os.environ.get("CFT_ATTENTION_SIMT") is not None      # the library reads the switch once, at load
GAP_EXP2 = 160.0                                             # exp2(-160) = 0 in fp32


# ---------------------------------------------------------------------------------------------- helpers
def _tc_chunks(dk):
    """(first column, width) of the head-dim chunks of the tcgen05 kernel (csrc/attention_tcgen05.cu): 64 / 32 / 16
    wide, widest first; a last chunk of 16 may cover the final 8 columns."""
    out, off = [], 0
    while off < dk:
        rem = dk - off
        w = 64 if rem >= 64 else (32 if rem >= 32 else 16)
        out.append((off, w))
        off += w
    return out


def _path(t, dk):
    """The kernel cft_attention runs for (T, dk), or None when it must refuse the shape."""
    if not SIMT and t == T and 16 <= dk <= 256 and len(_tc_chunks(dk)) <= 4:
        return "tcgen05"
    return "simt" if 3 * 128 * (dk + 2) * 2 + 128 * 129 * 4 <= 220 * 1024 else None


def _c_for(dk):
    """Smallest integer c with 2 c^2 log2(e) / sqrt(dk) >= 160: every key but the peak gets exp2(<= -160) = 0."""
    c = 1
    while 2 * c * c * LOG2E / math.sqrt(dk) < GAP_EXP2:
        c += 1
    return c


def _bf16_exact(t):
    return bool(torch.equal(t.double(), t.to(torch.bfloat16).double()))


def _peak_p(mx, dk):
    """The kernels' P of the peak score mx (float64 array): exp2f(fmaf(mx, scale, -mx * scale)) rounded to bf16 -- the
    tcgen05 kernels (attention_tcgen05.cu, cft_block.cu); returns (P in fp32 before rounding, P in bf16)."""
    scale = np.float32(np.float32(1.4426950408889634) / np.sqrt(np.float32(dk)))
    mx32 = np.asarray(mx, dtype=np.float32)
    mxs = (mx32 * scale).astype(np.float32)
    arg = (mx32.astype(np.float64) * np.float64(scale) - mxs.astype(np.float64)).astype(np.float32)   # fmaf: one rounding
    e = np.exp2(arg.astype(np.float64)).astype(np.float32)
    p = torch.from_numpy(e.astype(np.float32)).to(torch.bfloat16).double().numpy()
    return e, p


def _check_scores(S, dk, uniform, large=False):
    """S: float64 [..., T, T] exact scores.  Asserts the conditions under which the kernels' softmax is exact: partial
    sums below 2^24 (|S| <= c^2 dk bounds every partial sum), the gap to the second distinct score, and P of the peak
    rounding to exactly 1 in bf16 (or, for large logits, to a value p with bf16(fp32(p v) * fp32(1 / p)) = v)."""
    amax = float(S.abs().max())
    assert amax < 2 ** 24, amax
    mx = S.amax(-1, keepdim=True)
    if not uniform.all():
        below = torch.where(S < mx, S, torch.full_like(S, -math.inf)).amax(-1)
        gap = (mx.squeeze(-1) - below)[~uniform]
        gap_min = float(gap.min())
        assert gap_min * LOG2E / math.sqrt(dk) >= GAP_EXP2, (dk, gap_min)
    e, p = _peak_p(mx.numpy(), dk)
    if not large:
        assert (p == 1.0).all() and (np.abs(e.astype(np.float64) - 1.0) < 2.0 ** -10).all(), (dk, amax)
        return
    assert amax > 5e6 and (p != 1.0).any(), "large-logit case must take P of the peak away from 1"
    pv = np.unique(p)
    v = np.arange(-16, 17, dtype=np.float32)
    for pk in pv.astype(np.float32):                       # sum = p (one key), O = p v, out = O * (1 / sum)
        o = (pk * v).astype(np.float32) * (np.float32(1.0) / pk)
        assert torch.equal(torch.from_numpy(o).to(torch.bfloat16).float(), torch.from_numpy(v)), pk


def _softmax_exact(S, v):
    """The exact answer when every key below the peak gets P = 0 and every key at the peak P = 1: the mean of v over the
    keys that reach the row's maximum, rounded to bf16 (S float64 [..., Tq, Tk], v [..., Tk, dk])."""
    m = (S == S.amax(-1, keepdim=True)).double()
    return ((m @ v) / m.sum(-1, keepdim=True)).to(torch.bfloat16).double()


# ---------------------------------------------------------------------------------------------- 1. per-op attention
def _bit_columns(dk):
    """Column p of a head's code carries index bit bit_of[p]: bit 0 the first 8 columns (all of a 16-column head's first
    half); bits 1..6 are dealt to the other tcgen05 chunks (the rest of chunk 0 counts as one) so that each chunk holds
    bits no other chunk holds.  dk = 8: one bit per column, the last column constant (-1)."""
    if dk == 8:
        return list(range(7)) + [-1]
    chunks = _tc_chunks(dk) if len(_tc_chunks(dk)) <= 4 else [(0, dk)]
    groups = [(8, min(dk, chunks[0][0] + chunks[0][1]))] + [(o, min(dk, o + w)) for o, w in chunks[1:]]
    groups = [g for g in groups if g[1] > g[0]]
    bit_of = [0] * dk
    for gi, (lo, hi) in enumerate(groups):
        bits = [b for b in range(1, 7) if (b - 1) % len(groups) == gi]
        for p in range(lo, hi):
            bit_of[p] = bits[(p - lo) % len(bits)]
    assert sorted(set(bit_of)) == list(range(7))
    return bit_of


def _codes(idx, dk, base):
    """+-1 codes [n, dk] of the indices idx: base[p] * (-1)^(bit bit_of[p] of the index)."""
    bit_of = torch.tensor(_bit_columns(dk))
    bits = (idx[:, None] >> bit_of.clamp(min=0)[None, :]) & 1
    bits[:, bit_of < 0] = 0
    return base[None, :] * (1 - 2 * bits).double()


def attention_case(B, t, heads, dk, seed, groups=None, c=None):
    """qkv (float64 [B*t, 3C]) and the expected output (float64 [B*t, C]).  groups[h] = keys per code of head h:
    1 = hard attention (query -> one key), 2 .. 64 = tied keys, T = uniform (q = 0).  Checks the exactness conditions."""
    g = torch.Generator().manual_seed(seed)
    C = heads * dk
    large = c is not None
    c = c if large else _c_for(dk)
    assert _bf16_exact(torch.tensor([float(c)]))
    groups = groups or [1] * heads
    q = torch.zeros(B, heads, t, dk, dtype=torch.float64)
    k = torch.zeros_like(q)
    v = torch.randint(-16, 17, (B, heads, t, dk), generator=g).double()
    uniform = torch.zeros(B, heads, t, dtype=torch.bool)
    for b in range(B):
        for h in range(heads):
            gs = groups[h]
            base = (torch.randint(0, 2, (dk,), generator=g) * 2 - 1).double()
            key_idx = torch.randperm(t, generator=g) // gs                     # key s carries code key_idx[s]
            k[b, h] = c * _codes(key_idx, dk, base)
            if gs >= t:
                uniform[b, h] = True                                           # q = 0: every key scores 0
                continue
            tgt = torch.randperm(t, generator=g) // gs                         # query t wants code tgt[t]
            q[b, h] = c * _codes(tgt, dk, base)
            if gs == 1 and t == T:                                             # targets in both 64-key halves
                hit = (key_idx[None, :] == tgt[:, None]).double().argmax(1)
                assert (hit < 64).any() and (hit >= 64).any()
    S = q @ k.transpose(-1, -2)
    _check_scores(S, dk, uniform, large)
    ref = _softmax_exact(S, v)                                                 # [B, heads, t, dk]
    qkv = torch.cat([x.permute(0, 2, 1, 3).reshape(B * t, C) for x in (q, k, v)], 1)
    assert _bf16_exact(qkv)
    return qkv, ref.permute(0, 2, 1, 3).reshape(B * t, C), (q, k, v)


def _overhang_changes(qkv, qkv_parts, B, t, heads, dk):
    """For dk = 8 (mod 16): would the output change if the last chunk read the 8 columns after each head of q and k
    (the next head; after the last q head the first k head, after the last k head the first v head) instead of zeros?
    Returns a [B, heads] bool tensor."""
    C = heads * dk
    q, k, v = qkv_parts
    rows = qkv.view(B, t, 3 * C)
    ext = []
    for part in (0, 1):
        e = torch.zeros(B, heads, t, 8, dtype=torch.float64)
        for h in range(heads):
            lo = part * C + (h + 1) * dk
            e[:, h] = rows[:, :, lo:lo + 8]
        ext.append(e)
    S = q @ k.transpose(-1, -2) + ext[0] @ ext[1].transpose(-1, -2)
    return (_softmax_exact(S, v) != _softmax_exact(q @ k.transpose(-1, -2), v)).flatten(2).any(-1)


def _run_attention(cft, qkv, B, t, C, heads):
    x = qkv.to(DEV, torch.bfloat16)
    out = cft.ops.attention(x, B, t, C, heads)
    torch.cuda.synchronize()
    return out.double().cpu()


def _expect_exact(cft, B, t, heads, dk, seed, groups=None, c=None):
    path = _path(t, dk)
    C = heads * dk
    qkv, ref, parts = attention_case(B, t, heads, dk, seed, groups, c)
    if path is None:
        n0 = cft._lib.launch_count()
        with pytest.raises(cft.CftError):
            _run_attention(cft, qkv, B, t, C, heads)
        assert cft._lib.launch_count() == n0, "a refused shape must not launch anything"
        return path
    if path == "tcgen05" and dk % 16 == 8 and heads > 1:
        # every head whose next head has a nonzero q: its bit-0 columns tie or flip this head's nearest keys
        need = [h for h in range(heads - 1) if (groups or [1] * heads)[h + 1] < T]
        changed = _overhang_changes(qkv, parts, B, t, heads, dk)
        assert need and changed[:, need].all(), changed
    got = _run_attention(cft, qkv, B, t, C, heads)
    if not torch.equal(got, ref):
        bad = (got != ref).view(B, t, heads, dk).any(-1)
        where = bad.nonzero()[:6].tolist()
        raise AssertionError(f"{path} B={B} T={t} heads={heads} dk={dk}: {int(bad.sum())}/{bad.numel()} (image, query, "
                             f"head) rows differ, e.g. {where}, max |d| {float((got - ref).abs().max()):g}")
    return path


MIXED = [1, 2, 4, 8, 16, 32, 64, T]        # keys per code of heads 0, 1, 2, ...: hard, tied, uniform


@pytest.mark.parametrize("heads", [1, 3])
@pytest.mark.parametrize("dk", list(range(16, 257, 8)))
def test_per_op_attention_every_head_dim(dk, heads, cft):
    for B in (1, 3):
        hard = _expect_exact(cft, B, T, heads, dk, seed=dk * 10 + heads + B)
        tied = _expect_exact(cft, B, T, heads, dk, seed=dk * 10 + heads + B + 5000,
                             groups=[MIXED[(B + h + dk // 8) % len(MIXED)] for h in range(heads)])
        assert hard == tied
    print(f"\ndk={dk} heads={heads}: {hard or 'refused (CftError)'}"
          f"{' chunks ' + str([w for _, w in _tc_chunks(dk)]) if hard == 'tcgen05' else ''}")


@pytest.mark.parametrize("C", [128, 256, 320, 512, 640, 1024, 1280])
def test_per_op_attention_graph_widths(C, cft):
    """The (C, heads = 8) shapes of the model's CFT blocks; heads cycle through hard / tied / uniform attention."""
    for B in (1, 3):
        assert _expect_exact(cft, B, T, 8, C // 8, seed=C + B) is not None
        assert _expect_exact(cft, B, T, 8, C // 8, seed=C + B + 7, groups=MIXED) is not None


def test_per_op_attention_many_waves(cft):
    """B * heads = 640 CTAs: more than two waves of the tcgen05 kernel (two CTAs per SM)."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    B = 80
    assert B * 8 > 4 * n_sm
    _expect_exact(cft, B, T, 8, 32, seed=99, groups=[1, 1, 2, 1, 8, 1, 64, T])


@pytest.mark.parametrize("t", [1, 17, 64, 127])
@pytest.mark.parametrize("heads", [1, 3])
def test_per_op_attention_short_sequences_dk8(t, heads, cft):
    """T < 128 and dk = 8 run on the CUDA-core kernel only."""
    for dk in (8, 24):
        assert _expect_exact(cft, 3, t, heads, dk, seed=t * 7 + heads + dk) == "simt"


@pytest.mark.parametrize("dk", [16, 40, 64, 128])
def test_per_op_attention_large_logits(dk, cft):
    """max |S| ~ 1e7: the peak's P is no longer 1, yet p v / p rounds back to v."""
    c = int(math.sqrt(1e7 / dk))
    while not _bf16_exact(torch.tensor([float(c)])):
        c -= 1
    assert _expect_exact(cft, 2, T, 3, dk, seed=dk + 1, c=c) is not None


def test_per_op_attention_rejects_unsupported_shapes(cft):
    """Refused before any launch: CUDA-core shared memory above 220 KiB (T < 128 or more than 4 tensor-core chunks with
    dk > 200), a head dim that is not a multiple of 8, T outside [1, 128]."""
    x = torch.zeros(3 * 128, 3 * 256, dtype=torch.bfloat16, device=DEV)
    n0 = cft._lib.launch_count()
    for b, t, c, heads in ((3, 64, 256, 1), (1, 127, 208, 1), (1, 128, 248, 1), (1, 128, 100, 1), (1, 129, 64, 1),
                           (1, 0, 64, 1), (1, 128, 60, 3)):
        assert _path(t, c // heads) is None or (c // heads) % 8 or t > T or t < 1
        with pytest.raises(cft.CftError):
            cft.ops.attention(x, b, t, c, heads)
    torch.cuda.synchronize()
    assert cft._lib.launch_count() == n0


# ---------------------------------------------------------------------------------------------- 2. fused stack
HEADS = 8
LAYERS = 3


def _block_code(idx, dk):
    """Balanced +-1 codes [n, dk] of 7-bit indices: the 7 bits, their complements, then +1 / -1 padding pairs."""
    bits = ((idx[:, None] >> torch.arange(7)) & 1).double() * -2 + 1
    pad = torch.tensor([1.0, -1.0], dtype=torch.float64).repeat((dk - 14) // 2)
    return torch.cat([bits, -bits, pad.expand(idx.numel(), dk - 14)], 1)


def stack_tokens(B, d, seed):
    """x_in [B, 128, d]: row t = [a_t | b_t]; a-block j (dk wide) holds the code of pi_j(t), b-block j the code of
    pi_j(sigma_j(t)) -- per image, random permutations.  Returns x and sigma [B, 4, 128]."""
    dk = d // HEADS
    g = torch.Generator().manual_seed(seed)
    x = torch.zeros(B, T, d, dtype=torch.float64)
    sigma = torch.zeros(B, 4, T, dtype=torch.long)
    for b in range(B):
        for j in range(4):
            pi, sg = torch.randperm(T, generator=g), torch.randperm(T, generator=g)
            x[b, :, j * dk:(j + 1) * dk] = _block_code(pi, dk)
            x[b, :, d // 2 + j * dk:d // 2 + (j + 1) * dk] = _block_code(pi[sg], dk)
            sigma[b, j] = sg
    assert (x.sum(-1) == 0).all() and ((x * x).sum(-1) == d).all()          # mean 0, variance 1
    return x, sigma


def _sparse_pm1(rows, cols, nz, g):
    w = torch.zeros(rows, cols, dtype=torch.float64)
    for r in range(rows):
        w[r, torch.randperm(cols, generator=g)[:nz]] = (torch.randint(0, 2, (nz,), generator=g) * 2 - 1).double()
    return w


def stack_weights(d, kind, layer, seed):
    """Per-layer float64 parameters of a 3-layer stack: every Linear zero except layer `layer` of kind
    'attn' (hard attention), 'tied' (Wq = 0: uniform attention) or 'mlp'.  LN1 gamma = 1, beta = 0 (the codes pass
    unchanged); LN2 gamma in {1, 2}, beta in {0, +-0.5}."""
    dk = d // HEADS
    g = torch.Generator().manual_seed(seed)
    z = lambda *s: torch.zeros(*s, dtype=torch.float64)
    L = []
    for l in range(LAYERS):
        P = {"wqkv": z(3 * d, d), "bqkv": z(3 * d), "wo": z(d, d), "bo": z(d), "w1": z(4 * d, d), "b1": z(4 * d),
             "w2": z(d, 4 * d), "b2": z(d), "ln1_g": torch.ones(d, dtype=torch.float64), "ln1_b": z(d),
             "ln2_g": torch.randint(1, 3, (d,), generator=g).double(),
             "ln2_b": (torch.randint(-1, 2, (d,), generator=g) * 0.5).double()}
        if l == layer and kind in ("attn", "tied"):
            c = _c_for(dk)
            i = torch.arange(dk)
            for h in range(HEADS):
                j = h % 4
                if kind == "attn":
                    P["wqkv"][h * dk + i, d // 2 + j * dk + i] = c                 # q: b-block j
                P["wqkv"][d + h * dk + i, j * dk + i] = c                          # k: a-block j
            P["wqkv"][2 * d:] = _sparse_pm1(d, d, 8, g)                            # v
            P["bqkv"][2 * d:] = torch.randint(-8, 9, (d,), generator=g).double()
            perm = torch.randperm(d, generator=g)
            P["wo"][torch.arange(d), perm] = (torch.randint(0, 2, (d,), generator=g) * 2 - 1).double()
            P["bo"] = torch.randint(-8, 9, (d,), generator=g).double()
        elif l == layer:
            P["w1"] = _sparse_pm1(4 * d, d, 3, g)
            P["b1"] = torch.where(torch.rand(4 * d, generator=g) < 0.75, 32.0, -32.0).double()
            half = d // 2                                                         # W2: 8 nonzeros per row, one in
            for o in range(d):                                                    # each eighth of the hidden width
                for e in range(8):
                    P["w2"][o, e * half + (o * 7 + e * 13) % half] = float(torch.randint(0, 2, (1,), generator=g)) * 2 - 1
            P["b2"] = torch.randint(-8, 9, (d,), generator=g).double()
            read = (P["w2"] != 0).any(0) & (P["b1"] > 0)
            assert read.view(-1, 64).any(1).all(), "every 64 hidden columns must feed a nonzero W2 entry"
        L.append(P)
    return L


def _ln_exact(x, gamma, beta):
    """LayerNorm of balanced +-1 rows (mean 0, var 1): +-gamma * rsqrt(1 + eps) + beta, which rounds to +-gamma + beta in
    bf16 for the gamma, beta used here."""
    assert (x.abs() == 1).all() and (x.sum(-1) == 0).all(), "LayerNorm input must be balanced +-1 rows"
    y = x * gamma + beta
    assert (y != 0).all() and _bf16_exact(y)
    assert torch.equal((x / math.sqrt(1 + 1e-5) * gamma + beta).to(torch.bfloat16).double(), y)
    return y


def stack_reference(x, L):
    """float64 x after every layer ([layers] of [B, 128, d]); asserts the exactness conditions of each nonzero part."""
    B, _, d = x.shape
    dk = d // HEADS
    xs = []
    for P in L:
        if P["wqkv"].any():
            y = _ln_exact(x, P["ln1_g"], P["ln1_b"])
            qkv = y @ P["wqkv"].t() + P["bqkv"]
            assert _bf16_exact(qkv) and float((y.abs() @ P["wqkv"].abs().t()).max()) < 2 ** 24
            q, k, v = (qkv[..., i * d:(i + 1) * d].view(B, T, HEADS, dk).transpose(1, 2) for i in range(3))
            S = q @ k.transpose(-1, -2)
            _check_scores(S, dk, (S == 0).all(-1))
            att = _softmax_exact(S, v).transpose(1, 2).reshape(B, T, d)
            x = x + (att @ P["wo"].t() + P["bo"])
        if P["w1"].any():
            y = _ln_exact(x, P["ln2_g"], P["ln2_b"])
            pre = y @ P["w1"].t() + P["b1"]
            assert (pre.abs() >= 24).all() and _bf16_exact(pre)       # gelu_fast / erff give v or -0 exactly
            hid = pre.clamp(min=0)
            x = x + (hid @ P["w2"].t() + P["b2"])
            assert float(x.abs().max()) < 2 ** 20
        xs.append(x)
    return xs


def _load(g, L):
    """Write the float64 parameters into the GPT module (every value bf16-exact)."""
    with torch.no_grad():
        for blk, P in zip(g.trans_blocks, L):
            sa = blk.sa
            d = P["wo"].shape[0]
            for m, w, b in ((sa.que_proj, P["wqkv"][:d], P["bqkv"][:d]), (sa.key_proj, P["wqkv"][d:2 * d], P["bqkv"][d:2 * d]),
                            (sa.val_proj, P["wqkv"][2 * d:], P["bqkv"][2 * d:]), (sa.out_proj, P["wo"], P["bo"]),
                            (blk.mlp[0], P["w1"], P["b1"]), (blk.mlp[2], P["w2"], P["b2"])):
                assert _bf16_exact(w)
                m.weight.copy_(w.float())
                m.bias.copy_(b.float())
            blk.ln_input.weight.copy_(P["ln1_g"].float())
            blk.ln_input.bias.copy_(P["ln1_b"].float())
            blk.ln_output.weight.copy_(P["ln2_g"].float())
            blk.ln_output.bias.copy_(P["ln2_b"].float())


def _per_op(cft, x, w, B, d):
    """The same stack through per-op launches (LN -> QKV GEMM -> attention -> out GEMM with fp32 residual -> LN -> up
    GEMM + GELU -> down GEMM with fp32 residual): x after every layer."""
    ops = cft.ops
    x2d = x.view(B * T, d).clone()
    xs = []
    for L in w["layers"]:
        y = ops.layernorm(x2d, *L["ln1"])
        qkv = ops.gemm(y, L["qkv"][0], L["qkv"][1])
        att = ops.attention(qkv, B, T, d, HEADS)
        x2d = ops.gemm(att, L["out"][0], L["out"][1], residual=x2d, out_dtype=torch.float32)
        y = ops.layernorm(x2d, *L["ln2"])
        hid = ops.gemm(y, L["up"][0], L["up"][1], act=ops.ACT_GELU)
        x2d = ops.gemm(hid, L["down"][0], L["down"][1], residual=x2d, out_dtype=torch.float32)
        xs.append(x2d.view(B, T, d).clone())
    torch.cuda.synchronize()
    return xs


def _compare(got, want, what):
    for l, (a, b) in enumerate(zip(got, want)):
        a = a.double().cpu()
        if not torch.equal(a, b):
            bad = (a != b).any(-1)
            raise AssertionError(f"{what}: x after layer {l}: {int(bad.sum())}/{bad.numel()} token rows differ, e.g. "
                                 f"(image, token) {bad.nonzero()[:4].tolist()}, max |d| {float((a - b).abs().max()):g}")


KINDS = ("attn", "tied", "mlp")


def _stack_case(cft, d, B, kind, layer, seed):
    g = make_gpt(cft, d, LAYERS, seed=seed)
    L = stack_weights(d, kind, layer, seed)
    _load(g, L)
    x, _ = stack_tokens(B, d, seed + 1)
    want = stack_reference(x, L)
    assert not torch.equal(want[layer], x), "the nonzero layer must change x"
    return g, x.float().to(DEV), want


PLANS = [
    # d, cluster, B: every (DC, heads per CTA) instantiation of cft_gpt_block_kernel for heads = 8; B = 0: more images
    # than co-resident clusters (SMs // cluster + 3), so every cluster loops over images
    (128, 2, 2), (256, 4, 2), (256, 2, 3), (512, 4, 2), (256, 2, 0), (256, 4, 0),
]


@pytest.mark.parametrize("d,cluster,B", PLANS)
def test_fused_stack_bit_exact_per_layer(d, cluster, B, cft):
    if B == 0:
        B = torch.cuda.get_device_properties(0).multi_processor_count // cluster + 3
    for i, kind in enumerate(KINDS):
        layer = (i + d // 128 + cluster) % LAYERS
        g, x, want = _stack_case(cft, d, B, kind, layer, seed=d * 10 + cluster * 3 + i)
        w = g._weights(torch.device(DEV))
        dbg = torch.full((LAYERS, B, T, d), float("nan"), device=DEV)
        out = cft.ops.gpt_block(x, w["stack"], HEADS, cluster=cluster, debug_x=dbg)
        torch.cuda.synchronize()
        what = f"gpt_block d={d} cluster={cluster} B={B} {kind} layer {layer}"
        _compare(list(dbg), want, what)
        _ln_check(out.view(B * T, d), dbg[-1].view(B * T, d), g.ln_f.weight.detach(), g.ln_f.bias.detach(),
                  g.ln_f.eps, torch.zeros(B * T), what + " ln_f")
        _compare(_per_op(cft, x, w, B, d), want, what.replace("gpt_block", "per-op"))


@pytest.mark.parametrize("d", [128, 256, 320, 512, 640, 1024, 1280])
def test_per_op_stack_bit_exact_per_layer(d, cft):
    """LN -> GEMM -> attention -> GEMM per layer at every d of the graphs' CFT blocks."""
    B = 2
    for i, kind in enumerate(KINDS):
        layer = (i + d // 64) % LAYERS
        g, x, want = _stack_case(cft, d, B, kind, layer, seed=d * 10 + 7 + i)
        _compare(_per_op(cft, x, g._weights(torch.device(DEV)), B, d), want, f"per-op d={d} {kind} layer {layer}")
