"""GPU tests whose expected answer is known exactly (or to a bound derived from fp32), so that no tolerance scaled by the
largest output can hide an error:

1. Conv / GEMM launch plans.  Every conv and Linear of the s / l / x graphs (the catalogue of test_conv_plan_cpu.py at the
   image sizes and batches the model runs) is planned on the host; plans are grouped by the features that select code
   paths in the kernel (CTA pairs, tile shape, batch-spanning tiles, row reuse, resident weights, K unit, taps per stage,
   n-blocks and N tail, accumulator / staging layout, partial tiles in x / y / batch, stride, out dtype, residual) and the
   cheapest shape of each group runs.  Operands are integers in {-1, 0, 1}, each output channel sums a disjoint stride of
   the K = taps * Cin positions, bias and residual are integers of magnitude <= 8: every partial sum is an integer of
   magnitude <= 256, exact in bf16 and fp32, so the output must equal a float64 conv bit for bit.  The same shapes run
   through the CUDA-core reference kernel, with a chained 1x1, and with nonzero channel offsets into wider buffers.
2. Activation epilogues.  An identity GEMM turns every finite bf16 in [-40, 40] (plus 0, +-1e4, +-bf16 max) plus a
   per-column bias into the pre-activation v = fp32(x + b); |y - act(v)| (float64 act) must stay within the error bound
   that csrc/cft_common.cuh states for the active implementation, plus the rounding of the output.
3. LayerNorm at large offsets.  Rows with |mean| / std up to 1e4 through the per-op kernel and through the fused
   transformer stack (with zero Linear weights every layer leaves x unchanged and the output is ln_f(x)).  Tolerance
   |gamma| * (1e-5 + 2e-6 |mean| / sqrt(var + eps)): the mean is known to a few fp32 ulps of the offset, which is what
   the normalised output inherits; anything more comes from the variance."""
import ctypes as C
import math
import os

import pytest
import torch
import torch.nn.functional as F

from test_block_gpu import make_gpt
from test_conv_plan_cpu import _catalogue, _plan

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16_MAX = float(torch.finfo(torch.bfloat16).max)


# ---------------------------------------------------------------------------------------------- 1. conv / GEMM plans
def _graph_shapes():
    """(B, H, W, Cin, Cout real, Cout padded, k, s, out fp32, residual) of every conv / Linear launch of the graphs."""
    out = []
    for (hs, ws), batches in (((640, 640), (1, 2, 8, 32)), ((1024, 1280), (1,)), ((320, 416), (3,))):
        for cin, cout, k, s, lvl in _catalogue():
            sh = lvl - 1 if s == 2 else lvl
            f32 = cout in (24, 18, 42)                                  # Detect heads: fp32 output
            for B in batches:
                for res in ((False, True) if (k == 3 and s == 1 and cin == cout and lvl > 1) else (False,)):
                    out.append((B, hs >> sh, ws >> sh, cin, cout, (cout + 7) // 8 * 8, k, s, f32, res))   # C3 3x3 +- shortcut
    for d in (128, 256, 320, 512, 640, 1024, 1280):                     # GPT Linears (test_gpt_linear_shapes_get_valid_plans)
        for B in (1, 4, 32, 128):
            for cin, cout, f32 in ((d, 3 * d, False), (d, d, True), (d, 4 * d, False), (4 * d, d, True)):
                out.append((1, 1, 128 * B, cin, cout, cout, 1, 1, f32, f32))
    return out


def _signature(cft, shape):
    B, H, W, cin, _, cout, k, s, f32, res = shape
    p = _plan(cft, B, H, W, cin, cout, k, s, out_f32=f32, res=res)
    return (p.ctas, p.TW, p.TH, p.TB > 1, p.halo, p.b_res > 0, p.kelems, p.ups, p.kchunks > 1, p.block_n, p.n_blocks > 1,
            cout % p.block_n != 0, p.acc_stages, p.stage_c,
            p.Wo % p.TW != 0, p.Ho % p.TH != 0, B % p.TB != 0, s, f32, res)


def plan_representatives(cft):
    """{signature: the shape with the fewest MACs among those that get this plan signature}."""
    reps = {}
    for sh in _graph_shapes():
        B, H, W, cin, _, cout, k, s, _, _ = sh
        macs = B * ((H + s - 1) // s) * ((W + s - 1) // s) * cout * k * k * cin
        sig = _signature(cft, sh)
        if sig not in reps or macs < reps[sig][0]:
            reps[sig] = (macs, sh)
    return {sig: sh for sig, (_, sh) in reps.items()}


def _conv_args(cft, x, ldx, x_coff, shape, w, bias, y, ldy, y_coff, res=None, ldr=0, r_coff=0, chain=None):
    B, H, W, cin, _, cout, k, s, f32, _ = shape
    a = cft._lib.ConvArgs()
    a.x, a.B, a.H, a.W, a.Cin, a.ldx, a.x_coff = x.data_ptr(), B, H, W, cin, ldx, x_coff
    a.w, a.bias, a.Cout, a.k, a.stride, a.act = w.data_ptr(), bias.data_ptr(), cout, k, s, cft.ops.ACT_NONE
    a.res, a.ldr, a.r_coff = (res.data_ptr() if res is not None else None), ldr, r_coff
    a.y, a.ldy, a.y_coff, a.out_dtype, a.kw = y.data_ptr(), ldy, y_coff, (cft._lib.DT_F32 if f32 else cft._lib.DT_BF16), 0
    if chain is not None:                                   # (w2, bias2, y2, ldy2, y2_coff, act2, skip_y)
        w2, b2, y2, ldy2, y2_coff, act2, skip = chain
        a.w2, a.bias2, a.y2, a.ldy2, a.y2_coff, a.act2, a.skip_y = w2.data_ptr(), b2.data_ptr(), y2.data_ptr(), ldy2, \
            y2_coff, act2, int(skip)
    return a


def _run(cft, args, impl="tcgen05"):
    lib = cft._lib.lib()
    fn = lib.cft_conv2d if impl == "tcgen05" else lib.cft_conv2d_ref
    cft._lib.check(fn(C.byref(args), C.c_void_p(torch.cuda.current_stream().cuda_stream)), impl)


def _exact_operands(shape, seed):
    """x, w in {-1, 0, 1}; channel o of the Cout real ones owns the K positions o, o + Cout, o + 2 Cout, ... (padded
    channels stay zero, as pack_conv_weight leaves them); integer bias / residual in [-8, 8]."""
    B, H, W, cin, cout, cout_p, k, s, f32, res = shape
    g = torch.Generator().manual_seed(seed)
    K = k * k * cin
    Ho, Wo = (H + s - 1) // s, (W + s - 1) // s
    x = torch.randint(-1, 2, (B, H, W, cin), generator=g).float()
    w = torch.zeros(cout_p, K)
    pos = torch.arange(K)
    w[pos % cout, pos] = (torch.randint(0, 2, (K,), generator=g) * 2 - 1).float()
    bias = torch.zeros(cout_p)
    bias[:cout] = torch.randint(-8, 9, (cout,), generator=g).float()
    r = torch.randint(-8, 9, (B, Ho, Wo, cout_p), generator=g).float() if res else None
    bound = -(-K // cout) + 8 + (8 if res else 0)
    assert bound <= 256, (shape, bound)                     # every partial sum and output exact in bf16 and fp32
    odt = torch.float32 if f32 else torch.bfloat16
    return (x.to(DEV, torch.bfloat16), w.view(cout_p, k * k, cin).to(DEV, torch.bfloat16), bias.to(DEV),
            r.to(DEV, odt) if res else None, bound)


def _conv_f64(x, w, bias, k, s, res):
    """float64 reference on NHWC tensors (never TF32: the operands are converted to float64 first)."""
    cout_p = w.shape[0]
    cin = x.shape[-1]
    w64 = w.double().view(cout_p, k, k, cin).permute(0, 3, 1, 2)
    y = F.conv2d(x.double().permute(0, 3, 1, 2), w64, bias.double(), stride=s, padding=k // 2).permute(0, 2, 3, 1)
    return y + res.double() if res is not None else y


def _wide(t, lo, hi, fill):
    """t ([..., C]) at channels [lo, lo + C) of a buffer of lo + C + hi channels, the others set to `fill`."""
    buf = torch.full(t.shape[:-1] + (lo + t.shape[-1] + hi,), fill, dtype=t.dtype, device=t.device)
    buf[..., lo:lo + t.shape[-1]] = t
    return buf


def _chain_weight(cout, ymax, seed):
    """1x1 weight [Cout, 1, Cout] with as many +-1 per row as keep w2 . y + b2 within 256."""
    g = torch.Generator().manual_seed(seed)
    nz = max(1, min(8, (256 - 8) // ymax))
    w2 = torch.zeros(cout, cout)
    for o in range(cout):
        w2[o, torch.randperm(cout, generator=g)[:nz]] = (torch.randint(0, 2, (nz,), generator=g) * 2 - 1).float()
    b2 = torch.randint(-8, 9, (cout,), generator=g).float()
    assert nz * ymax + 8 <= 256
    return w2.view(cout, 1, cout).to(DEV, torch.bfloat16), b2.to(DEV)


def test_every_graph_plan_signature_is_bit_exact(cft):
    reps = plan_representatives(cft)
    print(f"\n{len(_graph_shapes())} graph launches -> {len(reps)} plan signatures")
    fails, n_chain, skip_done = [], 0, False
    for i, (sig, sh) in enumerate(sorted(reps.items(), key=lambda kv: str(kv[0]))):
        B, H, W, cin, cout, cout_p, k, s, f32, res = sh
        Ho, Wo = (H + s - 1) // s, (W + s - 1) // s
        odt = torch.float32 if f32 else torch.bfloat16
        x, w, bias, r, bound = _exact_operands(sh, seed=i)
        ref = _conv_f64(x, w, bias, k, s, r)
        what = f"B{B} {H}x{W} {cin}->{cout_p} k{k}s{s} {'f32' if f32 else 'bf16'}{' +res' if res else ''} sig={sig}"

        def check(got, tag):
            if not torch.equal(got.double(), ref):
                d = (got.double() - ref).abs()
                fails.append(f"{what} [{tag}]: {int((d > 0).sum())}/{d.numel()} differ, max |d| {float(d.max()):g}")

        y = torch.empty(B, Ho, Wo, cout_p, dtype=odt, device=DEV)
        for impl in ("tcgen05", "ref"):
            y.fill_(float("nan"))
            _run(cft, _conv_args(cft, x, cin, 0, sh, w, bias, y, cout_p, 0, r, cout_p, 0), impl)
            torch.cuda.synchronize()
            check(y, impl)
        # channel offsets into wider buffers: x at 8 of [8 | Cin | 16] (neighbours 3.0), y / residual at 16 of
        # [16 | Cout | 8]; the neighbouring channels must keep their sentinel
        xw = _wide(x, 8, 16, 3.0)
        yw = torch.full((B, Ho, Wo, cout_p + 24), -77.0, dtype=odt, device=DEV)
        rw = _wide(r, 16, 8, 5.0) if res else None
        _run(cft, _conv_args(cft, xw, cin + 24, 8, sh, w, bias, yw, cout_p + 24, 16, rw, cout_p + 24, 16))
        torch.cuda.synchronize()
        check(yw[..., 16:16 + cout_p], "coff")
        if not ((yw[..., :16] == -77).all() and (yw[..., 16 + cout_p:] == -77).all()):
            fails.append(f"{what} [coff]: channels next to the y slice were written")
        # the chained 1x1 (a Bottleneck's cv1 in the epilogue of its producer): y2 = w2 . bf16(y) + b2
        if cout_p in (64, 128) and not f32:
            n_chain += 1
            w2, b2 = _chain_weight(cout_p, bound, seed=1000 + i)
            ref2 = ref @ w2.double().view(cout_p, cout_p).t() + b2.double()
            skip = not skip_done
            skip_done = True
            y.fill_(float("nan"))
            y2 = torch.full((B, Ho, Wo, cout_p), float("nan"), dtype=odt, device=DEV)
            _run(cft, _conv_args(cft, x, cin, 0, sh, w, bias, y, cout_p, 0, r, cout_p, 0,
                                 chain=(w2, b2, y2, cout_p, 0, cft.ops.ACT_NONE, skip)))
            y2w = torch.full((B, Ho, Wo, cout_p + 16), -77.0, dtype=odt, device=DEV)
            yw.fill_(-77.0)
            _run(cft, _conv_args(cft, xw, cin + 24, 8, sh, w, bias, yw, cout_p + 24, 16, rw, cout_p + 24, 16,
                                 chain=(w2, b2, y2w, cout_p + 16, 8, cft.ops.ACT_NONE, False)))
            torch.cuda.synchronize()
            if skip:
                if not torch.isnan(y.float()).all():
                    fails.append(f"{what} [chain skip_y]: y was written")
            else:
                check(y, "chain y")
            for got, tag in ((y2, "chain y2" + (" skip_y" if skip else "")), (y2w[..., 8:8 + cout_p], "chain y2 coff")):
                if not torch.equal(got.double(), ref2):
                    d = (got.double() - ref2).abs()
                    fails.append(f"{what} [{tag}]: {int((d > 0).sum())}/{d.numel()} differ, max |d| {float(d.max()):g}")
            check(yw[..., 16:16 + cout_p], "chain y coff")
            if not ((y2w[..., :8] == -77).all() and (y2w[..., 8 + cout_p:] == -77).all()):
                fails.append(f"{what} [chain coff]: channels next to the y2 slice were written")
    print(f"plan signatures run: {len(reps)} (tcgen05, CUDA-core reference, channel offsets); chained 1x1: {n_chain}")
    assert skip_done and n_chain >= 2
    assert not fails, "\n".join(fails[:40])


# ---------------------------------------------------------------------------------------------- 2. activation epilogues
def _mantissa_bits(dtype):
    return {torch.bfloat16: 7, torch.float32: 23}[dtype]


def _half_ulp(a, dtype):
    tiny = torch.finfo(dtype).tiny
    e = torch.floor(torch.log2(a.clamp(min=tiny)))
    return torch.exp2(e - _mantissa_bits(dtype) - 1)


def _act64(v, act):
    if act == "none":
        return v
    if act == "silu":
        return v * torch.sigmoid(v)
    return 0.5 * v * torch.special.erfc(-v / math.sqrt(2.0))        # erf-GELU without cancellation in the tail


def _act_bound(v, act, impl):
    """The documented error of the fp32 activation at pre-activation v (csrc/cft_common.cuh)."""
    a = v.abs()
    if act == "none":
        return torch.zeros_like(v)
    if act == "silu":
        if impl == "ref":                                              # silu_f: __expf + __fdividef
            return (2.4 * a + 10.0) * 2.0 ** -24 * _act64(v, "silu").abs()
        if os.environ.get("CFT_SILU_EXP2"):                            # silu_fast: ex2 + rcp
            return (a + 8.0) * 2.0 ** -24 * _act64(v, "silu").abs()
        return 2.5e-4 * a                                              # silu_tanh: h + h tanh.approx(h)
    if impl == "ref" or os.environ.get("CFT_GELU_ERFF"):               # gelu_f: erff
        return 1.5e-7 * a
    return torch.full_like(v, 4e-7)                                    # gelu_fast: A&S erf through erfc


def _all_bf16_inputs():
    bits = torch.arange(-32768, 32768, dtype=torch.int32).to(torch.int16).view(torch.bfloat16).float()
    keep = torch.isfinite(bits) & (bits.abs() <= 40)
    extra = torch.tensor([0.0, 1e4, -1e4, BF16_MAX, -BF16_MAX]).to(torch.bfloat16).float()
    return torch.cat([bits[keep], extra])


ACT_CASES = [
    # act, out dtype, residual, impl
    *[(a, o, r, "tcgen05") for a in ("none", "silu", "gelu") for o in ("bf16", "f32") for r in (False, True)],
    *[(a, o, False, "ref") for a in ("silu", "gelu") for o in ("bf16", "f32")],
    ("silu", "bf16", True, "ref"),
    ("chain_silu", "bf16", False, "tcgen05"),
]


@pytest.mark.parametrize("act,out,res,impl", ACT_CASES)
def test_activation_epilogue_within_documented_bound(act, out, res, impl, cft):
    label = f"{act} {out}{' +res' if res else ''} {impl}"
    N = 264 if act != "chain_silu" else 128      # 264: two n-blocks (256 + a tail of 8); the chain needs 64 / 128
    vals = _all_bf16_inputs()
    M = -(-vals.numel() // N)
    a_mat = torch.zeros(M * N)
    a_mat[:vals.numel()] = vals
    a_mat = a_mat.view(M, N).to(DEV, torch.bfloat16)
    g = torch.Generator().manual_seed(3)
    bias = ((torch.arange(N) % 17) - 8).float() * torch.tensor([1.0, 0.5, 0.25])[torch.arange(N) % 3]
    bias[::5] = 0.0
    eye = torch.eye(N).view(N, 1, N).to(DEV, torch.bfloat16)
    odt = torch.float32 if out == "f32" else torch.bfloat16
    r = torch.randint(-8, 9, (M, N), generator=g).float().to(DEV, odt) if res else None
    code = {"none": 0, "silu": 1, "gelu": 2, "chain_silu": 0}[act]
    y = torch.empty(M, N, dtype=odt, device=DEV)
    shape = (1, 1, M, N, N, N, 1, 1, out == "f32", res)
    if act == "chain_silu":                       # y = x (act none, zero bias), y2 = SiLU(I . bf16(x) + b2)
        y2 = torch.empty(M, N, dtype=odt, device=DEV)
        zero = torch.zeros(N, device=DEV)
        args = _conv_args(cft, a_mat, N, 0, shape, eye, zero, y, N, 0,
                          chain=(eye, bias.to(DEV), y2, N, 0, cft.ops.ACT_SILU, False))
        args.act = code
        _run(cft, args)
        torch.cuda.synchronize()
        assert torch.equal(y, a_mat)
        y = y2
        act = "silu"
    else:
        args = _conv_args(cft, a_mat, N, 0, shape, eye, bias.to(DEV), y, N, 0, r, N if res else 0, 0)
        args.act = code
        _run(cft, args, impl)
        torch.cuda.synchronize()
    v = (a_mat.float() + bias.to(DEV)).double()                  # fp32(x + b): the kernel's pre-activation
    ref = _act64(v, act)
    if res:
        ref = ref + r.double()
    yd = y.double()
    m = torch.maximum(yd.abs(), ref.abs())
    tol = _act_bound(v, act, impl) + _half_ulp(m, torch.float32) + (_half_ulp(m, torch.bfloat16) if out == "bf16" else 0)
    err = (yd - ref).abs()
    assert torch.isfinite(yd).all()
    mask = torch.zeros(M * N, dtype=torch.bool)
    mask[:vals.numel()] = True
    mask = mask.view(M, N).to(DEV)
    av = v.abs()
    print(f"\n{label}: worst |y - act(v)| (ratio to the allowed error)")
    for lo, hi in ((0, 1), (1, 8), (8, 48), (48, math.inf)):
        sel = mask & (av >= lo) & (av < hi)
        if sel.any():
            print(f"  |v| in [{lo}, {hi}): {float(err[sel].max()):.3e} ({float((err / tol.clamp(min=1e-300))[sel].max()):.3f})")
    bad = mask & (err > tol)
    assert not bad.any(), (f"{int(bad.sum())} outputs beyond the documented bound, e.g. v = {v[bad][:4].tolist()} "
                           f"y = {yd[bad][:4].tolist()} ref = {ref[bad][:4].tolist()}")


# ---------------------------------------------------------------------------------------------- 3. LayerNorm
RATIOS = (0.0, 10.0, 100.0, 1e3, 1e4)
SIGMAS = (1e-3, 1.0, 1e3)
CONSTANTS = (0.0, 1.0, -3.7, 1234.5, -1e4)


def _ln_rows(n, C, seed):
    """n rows of C fp32 values: mean ratio * sigma, spread sigma for every (ratio, sigma), plus constant rows; returns the
    rows and each row's ratio (-1 for a constant row)."""
    g = torch.Generator().manual_seed(seed)
    kinds = [(r, s) for r in RATIOS for s in SIGMAS] + [(None, c) for c in CONSTANTS]
    rows, tags = [], []
    for i in range(n):
        r, s = kinds[i % len(kinds)]
        if r is None:
            rows.append(torch.full((C,), s, dtype=torch.float64))
            tags.append(-1.0)
        else:
            sign = 1.0 if (i // len(kinds)) % 2 == 0 else -1.0
            rows.append(sign * r * s + s * torch.randn(C, generator=g, dtype=torch.float64))
            tags.append(r)
    return torch.stack(rows).float(), torch.tensor(tags)


def _ln_check(y, x, gamma, beta, eps, tags, what):
    xd = x.double()
    ref = F.layer_norm(xd, (x.shape[-1],), gamma.double(), beta.double(), eps)
    mean, var = xd.mean(-1, keepdim=True), xd.var(-1, unbiased=False, keepdim=True)
    tol = gamma.double().abs() * (1e-5 + 2e-6 * mean.abs() / torch.sqrt(var + eps))
    err = (y.double() - ref).abs()
    ratio = (err / tol).amax(-1)
    tags = tags.to(ratio.device)
    print(f"\n{what}: worst |y - ref| (ratio to the tolerance) per |mean| / std")
    for r in (*RATIOS, -1.0):
        sel = tags == r
        if not sel.any():
            continue
        print(f"  {'constant' if r < 0 else f'{r:g}':>8}: {float(err[sel].max()):.3e} ({float(ratio[sel].max()):.3f})")
    worst = int(ratio.argmax())
    assert float(ratio.max()) <= 1.0, (f"{what}: row with |mean|/std {float(tags[worst]):g} off by "
                                       f"{float(err[worst].max()):.3e} ({float(ratio[worst]):.2f} x the tolerance)")


@pytest.mark.parametrize("C", [128, 256, 512])
def test_layernorm_at_large_offsets(C, cft):
    x, tags = _ln_rows(400, C, seed=C)
    g = torch.Generator().manual_seed(C + 1)
    gamma = torch.rand(C, generator=g) + 0.5
    beta = torch.randn(C, generator=g) * 0.1
    x, gamma, beta = x.to(DEV), gamma.to(DEV), beta.to(DEV)
    y = cft.ops.layernorm(x, gamma, beta, 1e-5, out_dtype=torch.float32)
    torch.cuda.synchronize()
    _ln_check(y, x, gamma, beta, 1e-5, tags, f"cft_layernorm C={C}")


@pytest.mark.parametrize("d,cluster", [(128, 0), (256, 0), (512, 0), (512, 4)])
def test_gpt_block_layernorm_at_large_offsets(d, cluster, cft):
    """Zero Linear weights and biases: every layer adds exactly 0 to x, so the stack returns ln_f(x_in) -- computed by the
    same in-kernel LayerNorm step as LN1 / LN2."""
    layers, B = 2, 3
    g = make_gpt(cft, d, layers, seed=d)
    with torch.no_grad():
        for m in g.modules():
            if isinstance(m, torch.nn.Linear):
                m.weight.zero_()
                m.bias.zero_()
    x, tags = _ln_rows(B * 128, d, seed=d + cluster)
    x = x.view(B, 128, d).to(DEV)
    w = g._weights(torch.device(DEV))["stack"]
    assert cft.ops.gpt_block_supported(B, d, g.h, 128)
    dbg = torch.full((layers, B, 128, d), float("nan"), device=DEV)
    out = cft.ops.gpt_block(x, w, g.h, cluster=cluster, debug_x=dbg)
    torch.cuda.synchronize()
    for l in range(layers):
        assert torch.equal(dbg[l], x), f"layer {l} changed x"
    _ln_check(out.view(B * 128, d), x.view(B * 128, d), g.ln_f.weight.detach(), g.ln_f.bias.detach(), g.ln_f.eps, tags,
              f"gpt_block ln_f d={d} cluster={cluster}")
