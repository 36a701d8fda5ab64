"""CPU suite: the host-side launch planner of ``cft_conv2d`` (tiling, CTA pairs, pipeline depth, shared-memory budget,
TMEM ring, epilogue staging) through ``cft_debug_conv_plan`` -- no device work.  Every conv / linear shape of the
yolov5{s,l,x}-x3 graphs (SURVEY.md section 8d catalogue at 640x640 and 1024x1280, batch 1..128) plus a dense grid of
other shapes must get a plan that satisfies the kernel's structural invariants."""
import ctypes as C
import itertools

import pytest

SMEM_MAX = 227 * 1024          # dynamic shared memory per CTA on sm_100
TMEM_COLS = 512


def _plan(cft, B, H, W, cin, cout, k, s, kw=0, out_f32=False, res=False):
    L = cft._lib
    lib = cft.load()
    a = L.ConvArgs()
    a.x, a.w, a.y = 0x100000, 0x200000, 0x300000            # never dereferenced by the planner
    a.bias, a.res = None, (0x400000 if res else None)
    a.B, a.H, a.W, a.Cin, a.ldx, a.x_coff = B, H, W, cin, cin, 0
    a.Cout, a.k, a.stride, a.act = cout, k, s, 1
    a.ldr, a.r_coff = (cout if res else 0), 0
    a.ldy, a.y_coff, a.out_dtype, a.kw = cout, 0, (1 if out_f32 else 0), kw
    p = L.ConvPlan()
    rc = lib.cft_debug_conv_plan(C.byref(a), C.byref(p))
    assert rc == 0, lib.cft_last_error().decode()
    return p


def _check(p, B, H, W, cin, cout, k, s, what, min_stages=2):
    ho, wo = (H + s - 1) // s, (W + s - 1) // s
    flat = k == 1 and s == 1 and (B > 1 or H > 1)                      # 1x1 convs are walked as one [B*H*W, C] matrix
    if flat:
        assert (p.Ho, p.Wo) == (1, B * H * W), what
        npix = B * H * W
        assert p.m_tiles * p.TW * p.TH >= npix and (p.m_tiles - 1) * p.TW * p.TH < npix, what
    else:
        assert (p.Ho, p.Wo) == (ho, wo), what
        assert p.tiles_x * p.TW >= wo and p.tiles_y * p.TH >= ho, what   # tiles cover the output
        assert (p.tiles_x - 1) * p.TW < wo and (p.tiles_y - 1) * p.TH < ho, what
        assert p.TB >= 1 and p.m_tiles == -(-B // p.TB) * p.tiles_x * p.tiles_y, what   # TB consecutive images per tile
        assert p.m_tiles <= B * -(-wo // min(wo, 128)) * -(-ho // max(1, min(ho, 128 // min(wo, 128)))), what   # never worse than rows
        if p.halo:
            assert p.TB == 1, what
    assert 1 <= p.TW * p.TH * p.TB <= 128, what                         # one UMMA M tile
    assert p.block_n % 16 == 0 and 16 <= p.block_n <= 256, what         # UMMA N constraint (M = 128)
    assert p.n_blocks * p.block_n >= cout and (p.n_blocks - 1) * p.block_n < cout, what
    assert p.ctas in (1, 2), what
    if p.ctas == 2:                                                     # cta_group::2: M = 256, N % 32 == 0
        assert p.block_n % 32 == 0 and p.kelems == 64 and p.m_tiles >= 2, what
    assert p.num_tiles == ((p.m_tiles + p.ctas - 1) // p.ctas) * p.n_blocks, what
    assert p.kelems in (16, 32, 64) and p.kchunks * p.kelems >= cin and (p.kchunks - 1) * p.kelems < cin, what
    assert p.acc_stages * p.acc_cols == TMEM_COLS and p.acc_cols >= p.block_n, what
    assert min_stages <= p.stages <= 8, what                            # a pipeline, within the barrier arrays
    if p.b_res:
        assert p.halo and p.ctas == 1 and p.n_blocks == 1 and p.stages >= 3 and p.b_slot == 0, what
        assert p.b_res >= 9 * p.kchunks * p.block_n * p.kelems * 2 and p.b_res <= 96 * 1024, what   # whole 3x3 weight matrix
    if p.halo:
        assert k == 3 and s == 1 and wo % 8 == 0 and ho % 16 == 0 and (p.TW, p.TH) == (8, 16), what
        assert p.a_slot >= p.ups * (p.TH + 2) * p.TW * p.kelems * 2, what
    else:
        assert p.a_slot >= 128 * p.kelems * 2 * (p.ups if p.ups > 1 else 1) or p.a_slot == 16384, what
    assert p.a_slot % 1024 == 0 and p.b_slot % 1024 == 0 and p.b_res % 1024 == 0, what   # swizzle-atom alignment
    assert p.teams in (1, 2) and p.stage_c in (8192, 16384), what
    assert p.smem_bytes <= SMEM_MAX, (what, p.smem_bytes)
    assert p.smem_bytes == 1024 + p.stages * (p.a_slot + p.b_slot) + p.b_res + 4 * p.stage_c + 3392, what
    assert 1 <= p.grid <= 148 and p.grid % p.ctas == 0, what


def _catalogue():
    """(Cin, Cout, k, s, level) of every conv / linear the three graphs launch (after the cv1||cv2 and QKV merges)."""
    shapes = set()
    for wm in (0.5, 1.0, 1.25):                                        # s / l / x width multiples
        c = lambda v: max(8, int(-(-v * wm // 8) * 8))                  # make_divisible(v * wm, 8)
        w = [c(64), c(128), c(256), c(512), c(1024)]                    # P1..P5 widths
        shapes.add((16, w[0], 3, 1, 1))                                 # Focus conv on the 16-channel gather
        for lvl in range(1, 5):
            cin, cout = w[lvl - 1], w[lvl]
            shapes.add((cin, cout, 3, 2, lvl + 1))                      # stride-2 downsampler
            h = cout // 2
            shapes.update({(cout, cout, 1, 1, lvl + 1), (h, h, 1, 1, lvl + 1), (h, h, 3, 1, lvl + 1)})   # C3
        shapes.update({(w[4], w[4] // 2, 1, 1, 5), (2 * w[4], w[4], 1, 1, 5)})          # SPP
        shapes.update({(w[4], w[3], 1, 1, 5), (w[3], w[2], 1, 1, 4), (w[4], w[3], 1, 1, 4), (w[3], w[2], 1, 1, 3),
                       (w[2], w[2], 3, 2, 4), (w[3], w[3], 3, 2, 5)})                   # PANet neck
        for no in (24, 18, 42):                                                          # Detect (nc 3 / 1 / 9)
            shapes.update({(w[2], no, 1, 1, 3), (w[3], no, 1, 1, 4), (w[4], no, 1, 1, 5)})
    return sorted(shapes)


@pytest.mark.parametrize("size,batches", [((640, 640), (1, 2, 8, 32, 128)), ((1024, 1280), (1, 8)), ((320, 416), (3,))])
def test_every_graph_shape_gets_a_valid_plan(cft, size, batches):
    n = 0
    for cin, cout, k, s, lvl in _catalogue():
        hin = size[0] >> (lvl - (1 if s == 2 else 0)) if s == 2 else size[0] >> lvl
        win = size[1] >> (lvl - (1 if s == 2 else 0)) if s == 2 else size[1] >> lvl
        for B in batches:
            cout_p = (cout + 7) // 8 * 8
            p = _plan(cft, B, hin, win, cin, cout_p, k, s, out_f32=cout in (24, 18, 42))
            _check(p, B, hin, win, cin, cout_p, k, s, f"{cin}->{cout} k{k}s{s} {hin}x{win} B{B}")
            n += 1
    assert n >= 90 * len(batches)


def test_gpt_linear_shapes_get_valid_plans(cft):
    for d in (128, 256, 320, 512, 640, 1024, 1280):
        for B in (1, 4, 32, 128):
            M = 128 * B
            for cin, cout, f32, res in ((d, 3 * d, False, False), (d, d, True, True), (d, 4 * d, False, False),
                                        (4 * d, d, True, True)):
                p = _plan(cft, 1, 1, M, cin, cout, 1, 1, out_f32=f32, res=res)
                _check(p, 1, 1, M, cin, cout, 1, 1, f"gemm M{M} K{cin} N{cout}")


def test_chained_1x1_keeps_every_channel_in_one_n_block(cft):
    """The chained 1x1 multiplies the whole Cout-wide tile of y: a layer with few tiles must not get its N split into
    n-blocks the way an unchained one does (1x1 producers and Cin <= 113 3x3 producers of 128 channels)."""
    L = cft._lib
    lib = cft.load()
    for B, H, W, cin, cout, k, s in ((3, 20, 26, 128, 128, 1, 1), (1, 1, 265, 128, 128, 1, 1), (1, 160, 160, 64, 128, 3, 2),
                                     (3, 80, 104, 64, 128, 3, 2), (2, 32, 32, 64, 64, 3, 1), (1, 20, 20, 128, 128, 3, 1)):
        unchained = _plan(cft, B, H, W, cin, cout, k, s)
        a = L.ConvArgs()
        a.x, a.w, a.y, a.w2, a.y2 = 0x100000, 0x200000, 0x300000, 0x400000, 0x500000
        a.B, a.H, a.W, a.Cin, a.ldx = B, H, W, cin, cin
        a.Cout, a.k, a.stride, a.act, a.act2, a.ldy, a.ldy2 = cout, k, s, 1, 1, cout, cout
        p = L.ConvPlan()
        assert lib.cft_debug_conv_plan(C.byref(a), C.byref(p)) == 0, lib.cft_last_error().decode()
        what = f"{cin}->{cout} k{k}s{s} {H}x{W} B{B} (unchained block_n {unchained.block_n})"
        assert p.n_blocks == 1 and p.block_n == cout and p.num_tiles * p.ctas >= p.m_tiles, what


def test_plan_grid_of_shapes(cft):
    """Dense grid: every combination must either plan validly or be rejected with CFT_E_ARG -- never plan garbage."""
    L = cft._lib
    n_ok = 0
    for cin, cout, (k, s), (H, W), B in itertools.product(
            (8, 16, 24, 32, 48, 64, 80, 96, 128, 160, 192, 256, 320, 384, 512, 640, 1024, 1280, 2048),
            (8, 16, 24, 40, 64, 80, 96, 128, 160, 256, 320, 512, 640, 1024, 1280),
            ((1, 1), (3, 1), (3, 2)),
            ((160, 160), (80, 80), (40, 40), (20, 20), (12, 20), (128, 160), (6, 6), (2, 2)),
            (1, 5, 32)):
        p = _plan(cft, B, H, W, cin, cout, k, s)
        # off-graph corner (row-reuse mode, Cin <= 64 with Cout >= 256: three weight taps of a 256-wide tile per stage)
        # may get a single-stage ring: slow but functional; every shape of the real graphs has >= 2 (tests above)
        _check(p, B, H, W, cin, cout, k, s, f"{cin}->{cout} k{k}s{s} {H}x{W} B{B}", min_stages=1)
        n_ok += 1
    assert n_ok > 10000


def test_plan_rejects_bad_arguments(cft):
    L = cft._lib
    lib = cft.load()
    a = L.ConvArgs()
    a.x, a.w, a.y = 0x100000, 0x200000, 0x300000
    a.B, a.H, a.W, a.Cin, a.ldx = 1, 8, 8, 12, 12                      # Cin not a multiple of 8
    a.Cout, a.k, a.stride, a.act, a.ldy = 16, 3, 1, 1, 16
    p = L.ConvPlan()
    assert lib.cft_debug_conv_plan(C.byref(a), C.byref(p)) == 1        # CFT_E_ARG
    assert b"multiples of 8" in lib.cft_last_error()
    a.Cin, a.ldx, a.k = 16, 16, 5
    assert lib.cft_debug_conv_plan(C.byref(a), C.byref(p)) == 1
    a.k, a.stride = 1, 2
    assert lib.cft_debug_conv_plan(C.byref(a), C.byref(p)) == 1        # stride 2 only for 3x3
    assert lib.cft_debug_conv_plan(C.byref(a), None) == 1


def test_batch_spanning_tiles_are_exact_on_40x40_and_20x20(cft):
    """40 x 40 and 20 x 20 maps have no waste-free 2-D tile of 128 pixels; tiles of 8 x 8 x 2 images / 4 x 4 x 8 images
    (or any other exact (TW, TH, TB)) fill every UMMA row: batch 32 -> 400 / 100 tiles instead of 448 / 128."""
    for (H, W, cin, cout, s, want) in [(40, 40, 256, 256, 1, 400), (20, 20, 512, 512, 1, 100), (80, 80, 256, 512, 2, 400),
                                       (40, 40, 512, 1024, 2, 100)]:
        p = _plan(cft, 32, H, W, cin, cout, 3, s)
        assert p.m_tiles == want and p.TW * p.TH * p.TB == 128, (H, W, p.TW, p.TH, p.TB, p.m_tiles)
        _check(p, 32, H, W, cin, cout, 3, s, f"{H}x{W}")
    p = _plan(cft, 1, 40, 40, 256, 256, 3, 1)                # batch 1: nothing to span
    assert p.TB == 1 and p.m_tiles == 14
    p = _plan(cft, 3, 20, 20, 512, 512, 3, 1)                # ragged batch: 3 images in one 4 x 8 x 3 ... tile set
    assert p.TW * p.TH * p.TB <= 128 and p.m_tiles <= 12
