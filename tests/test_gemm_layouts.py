"""-m gpu: the tcgen05 GEMM (gemm::launch through b200seg_gemm_run) in every output layout, sharing geometry, tile width and
switch setting, against an fp64 reference of the same bf16 operands.

Every case runs on views into larger allocations: operands at a 16-byte offset with a row pitch above their logical width, the
padding and everything around them bf16 NaN (a tensor map that reads past the logical extent turns the result NaN); outputs with
padded rows, gaps between images and guard bands, the logical footprint pre-filled with NaN (an unwritten element is caught) and
everything else with a sentinel bit pattern that must survive the launch.

Two tiers of data:
  * exact: operands are integers in [-8, 8], K <= 2^14, so every partial sum is an integer below 2^24 and the fp32 result is exact
    in any summation order -- every layout must equal the reference bit for bit, whatever the geometry, tile width or split (SEAM:
    power-of-two scales, dyadic bias / identity, so the fp32 tail is exact too and the bf16 output pins round-to-nearest-even);
  * accuracy: bf16-rounded normals, each element within TAU * sum_k |a_ik b_kj| of the reference.
Each launch also checks the kernel launch() picked against POLICY below (the semantics b200seg.h documents for the switches)."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

F32, COLS, ROWS, BF16, SEAM, STATS = range(6)
LAYOUT_NAMES = {F32: "f32", COLS: "f32_nchw_cols", ROWS: "f32_nchw_rows", BF16: "bf16", SEAM: "seam", STATS: "f32_nchw_rows_stats"}
NONE, SB, SA, PAIR = 0, 1, 2, 4          # sharing geometries (gemm_sm100.cuh SHARE_*)
ERR_ARG = 1
GUARD = 64                                # elements of guard band before and after every output (a multiple of 8: keeps bf16 alignment)
F32_NAN, BF16_NAN = 0x7FC00000, 0x7FC0
F32_SENTINEL, BF16_SENTINEL = 0x7FA5A5A5, 0x7FA5     # NaN bit patterns no kernel produces: compared as integers
# accuracy tier: |D - ref| <= TAU * sum_k |a_ik b_kj|; about 4x the worst ratio measured on a B200 (1000 W): 6.2e-7 for
# F32_NCHW_ROWS, 4.4e-7 for F32_NCHW_COLS, 4.2e-7 for F32 (BF16 and the STATS c are pinned to F32 / F32_NCHW_ROWS below)
TAU = 2.5e-6
# the switches as the library sets them when it loads (_lib.load() applies these variables)
LOAD_TIME = dict(sharing=int(os.environ.get("B200SEG_GEMM_SHARING") or 1), narrow=int(os.environ.get("B200SEG_GEMM_NARROW") or 1),
                 dgrad=1, fwd=1)


def cdiv(a, b):
    return -(-a // b)


@pytest.fixture(scope="module")
def lib():
    from rnd_semantic_segmentation_b200 import _lib
    _lib.load()
    yield _lib
    set_switches(_lib)                    # every setter also drops the step-graph cache: no later test inherits a mode


def set_switches(lib, **kw):
    """Set all four GEMM switches (unnamed ones to their load-time value); returns the setting."""
    s = dict(LOAD_TIME, **kw)
    lib.gemm_set_sharing(s["sharing"])
    lib.gemm_set_narrow_tiles(s["narrow"])
    lib.gemm_set_dgrad_mode(s["dgrad"])
    lib.gemm_set_fwd_mode(s["fwd"])
    return s


# ------------------------------------------------------------------ the kernel-choice policy of launch()
def clamp_splits(K, splits):
    kb = cdiv(K, 64)
    s = max(1, min(splits, kb))
    per = cdiv(kb, s)
    return cdiv(kb, per), per


def policy(layout, M, N, K, splits, a_mn, b_mn, share, fallback, sw, sms):
    """The variant launch() must pick (b200seg.h: b200seg_gemm_set_sharing / _narrow_tiles / _dgrad_mode): mode 0 = one CTA per
    tile, 3 = multicast-B pairs as cta_group::2, 4 = every shared geometry as cta_group::2, 5 = no cta_group::2 (the caller's
    fallback); STATS is always a pair; a pair needs two tiles along its dimension (STATS excepted); the 224 / 192-column tiles
    only for K-major operands, fp32 output and unshared B, when they cut rounds x columns; the register-store kernel for the
    rows layouts on cta_group::2 pairs with K-major B, except under dgrad mode 2 (streaming stores, the generic kernel)."""
    mode = sw["sharing"]
    s = share
    if mode == 0:
        s = NONE
    if mode == 3 and s == SB:
        s = PAIR
    if mode == 4 and s in (SA, SB):
        s = PAIR
    if mode == 5 and s == PAIR:
        s = fallback
    if layout == STATS:
        s = PAIR
    mt, nt = cdiv(M, 128), cdiv(N, 256)
    if s == SB and mt < 2:
        s = NONE
    if s == PAIR and mt < 2 and layout != STATS:
        s = NONE
    if s == SA and nt < 2:
        s = NONE
    bn = 256
    if sw["narrow"] and not a_mn and not b_mn and layout not in (BF16, SEAM) and s in (NONE, SA):
        used, _ = clamp_splits(K, splits)
        workers = sms // 2 if s == SA else sms
        best = None
        for cand in (256, 224, 192):
            ntc = cdiv(N, cand)
            if s == SA and ntc < 2:
                continue
            cost = cdiv(mt * (cdiv(ntc, 2) if s == SA else ntc) * used, workers) * cand
            if best is None or cost < best:
                best, bn = cost, cand
    row_hw = (2 if sw["dgrad"] == 2 else 1) if layout == ROWS else (1 if layout == STATS else 0)
    rs = row_hw == 1 and s == PAIR and not b_mn
    return dict(a_mn=int(a_mn), b_mn=int(b_mn), share=s, bn=bn, rs=int(rs), seam=int(layout == SEAM), stats=int(layout == STATS))


# ------------------------------------------------------------------ buffers
def exact_values(rows, cols, g):
    return torch.randint(-8, 9, (rows, cols), generator=g).float()


def random_values(rows, cols, g):
    return torch.randn(rows, cols, generator=g).to(torch.bfloat16).float()


def operand(vals, mn):
    """vals [rows][K] (bf16-representable) -> a bf16 view of the operand as the GEMM reads it (K-major [rows][K] or MN-major
    [K][rows]) at a 16-byte offset into a NaN-filled allocation, pitch above the logical width; returns (view, pitch)."""
    logical = vals.t() if mn else vals
    R, C = logical.shape
    pitch = cdiv(C, 8) * 8 + 8
    buf = torch.full((8 + R * pitch + 64,), float("nan"), dtype=torch.bfloat16, device="cuda")
    view = buf[8:8 + R * pitch].view(R, pitch)[:, :C]
    view.copy_(logical.to(torch.bfloat16))
    return view, pitch


class Output:
    """The output buffer of one launch: footprint index map, NaN-filled footprint, sentinel everywhere else."""

    def __init__(self, layout, M, N, splits, hw=0, off4=False, single_plane=False):
        self.layout, self.M, self.N = layout, M, N
        bf16 = layout in (BF16, SEAM)
        self.row_stride = self.img_stride = self.split_stride = 0
        m = torch.arange(M, device="cuda").view(M, 1)
        n = torch.arange(N, device="cuda").view(1, N)
        if layout in (F32, BF16):
            self.row_stride = cdiv(N, 8) * 8 + 8 + (1 if off4 else 0)
            idx = m * self.row_stride + n
            self.split_stride = M * self.row_stride + (8 if bf16 else (3 if off4 else 4))
        elif layout == COLS:
            self.row_stride = hw + (5 if off4 else 4)
            self.img_stride = M * self.row_stride + (3 if off4 else 4)
            idx = torch.div(n, hw, rounding_mode="floor") * self.img_stride + m * self.row_stride + n % hw
            self.split_stride = cdiv(N, hw) * self.img_stride + (3 if off4 else 8)
        elif layout in (ROWS, STATS):
            self.img_stride = 0 if single_plane else N * hw + 3            # an odd gap between images
            idx = torch.div(m, hw, rounding_mode="floor") * self.img_stride + n * hw + m % hw
        else:                                                              # SEAM: plain [M][N]
            idx = m * N + n
        self.idx = idx.view(1, M, N) + torch.arange(splits, device="cuda").view(splits, 1, 1) * self.split_stride
        self.base = GUARD + (1 if off4 and not bf16 else 0)
        total = self.base + int(self.idx.max()) + 1 + GUARD
        self.bits = torch.full((total,), BF16_SENTINEL if bf16 else F32_SENTINEL, dtype=torch.int16 if bf16 else torch.int32,
                               device="cuda")
        self.sentinel = self.bits[0].item()
        self.bits[self.base + self.idx.flatten()] = BF16_NAN if bf16 else F32_NAN
        self.dtype = torch.bfloat16 if bf16 else torch.float32
        self.origin = self.bits[self.base:].view(self.dtype)

    def values(self):
        """[splits][M][N] as written; asserts the footprint has no NaN left and nothing outside it changed."""
        d = self.bits[self.base + self.idx].view(self.dtype)
        outside = torch.ones_like(self.bits, dtype=torch.bool)
        outside[self.base + self.idx.flatten()] = False
        changed = int((self.bits[outside] != self.sentinel).sum())
        assert changed == 0, f"{changed} elements written outside the output footprint"
        nan = int(torch.isnan(d).sum())
        assert nan == 0, f"{nan} of {d.numel()} output elements NaN (unwritten, or an operand read past its extent)"
        return d


class Stats:
    """float2 [ceil(M / 32)][N] with the same NaN footprint / sentinel guard scheme."""

    def __init__(self, M, N):
        self.G = cdiv(M, 32)
        self.bits = torch.full((2 * (GUARD + self.G * N + GUARD),), F32_SENTINEL, dtype=torch.int32, device="cuda")
        self.bits[2 * GUARD:2 * (GUARD + self.G * N)] = F32_NAN
        self.origin = self.bits[2 * GUARD:].view(torch.float32)
        self.N = N

    def values(self):
        inner = self.bits[2 * GUARD:2 * (GUARD + self.G * self.N)]
        assert bool((self.bits[:2 * GUARD] == F32_SENTINEL).all()) and bool((self.bits[2 * (GUARD + self.G * self.N):] == F32_SENTINEL).all()), \
            "statistics written outside [ceil(M / 32)][N]"
        v = inner.view(torch.float32).view(self.G, self.N, 2).double()
        assert not bool(torch.isnan(v).any()), "statistics left unwritten"
        return v[..., 0], v[..., 1]


def seam_inputs(M, N, hw, g, exact=True):
    """scale (power of two), bias (k / 4), identity (k / 8, fp32 NCHW [n_img][N][hw]; pixels past M NaN)."""
    scale = torch.tensor([0.25, 0.5, 1.0, 2.0])[torch.randint(0, 4, (N,), generator=g)]
    bias = torch.randint(-64, 65, (N,), generator=g).float() / 4
    n_img = cdiv(M, hw)
    ident = torch.randint(-256, 257, (n_img, N, hw), generator=g).float() / 8
    flat = ident.permute(0, 2, 1).reshape(n_img * hw, N)
    flat[M:] = float("nan")
    ident = flat.view(n_img, hw, N).permute(0, 2, 1).contiguous()
    return scale.cuda(), bias.cuda(), ident.cuda()


def seam_reference(acc, scale, bias, ident, M, hw):
    N = acc.shape[1]
    idm = ident.permute(0, 2, 1).reshape(-1, N)[:M].double()
    return torch.relu(acc * scale.double() + bias.double() + idm)


def group_stats(c, M):
    """fp64 (mean, M2) and sum v^2 of c [M][N] per 32-row group."""
    G = cdiv(M, 32)
    pad = torch.zeros(G * 32, c.shape[1], dtype=torch.float64, device=c.device)
    pad[:M] = c
    cnt = torch.tensor([min(32, M - 32 * i) for i in range(G)], dtype=torch.float64, device=c.device).view(G, 1)
    v = pad.view(G, 32, -1)
    mask = (torch.arange(G * 32, device=c.device) < M).double().view(G, 32, 1)
    mean = v.sum(1) / cnt
    m2 = (((v - mean.unsqueeze(1)) * mask) ** 2).sum(1)
    return mean, m2, (v * v).sum(1), cnt


# ------------------------------------------------------------------ one launch
class Run:
    pass


def run_case(lib, layout, M, N, K, *, splits=1, a_mn=False, b_mn=False, hw=0, share=NONE, fallback=SB, sw=None, exact=True,
             seed=0, off4=False, single_plane=False, sm_reserve=0, data=None, check_policy=True):
    """Launches one GEMM, checks footprint / sentinels / clamp / kernel choice; returns a Run with the values and references."""
    sw = sw or LOAD_TIME
    g = torch.Generator().manual_seed(seed)
    if data is None:
        gen = exact_values if exact else random_values
        A, B = gen(M, K, g).cuda(), gen(N, K, g).cuda()
        extra = seam_inputs(M, N, hw, g) if layout == SEAM else None
    else:
        A, B, extra = data
    av, ap = operand(A, a_mn)
    bv, bp = operand(B, b_mn)
    want_splits, per = clamp_splits(K, splits)
    out = Output(layout, M, N, want_splits, hw, off4, single_plane)
    st = Stats(M, N) if layout == STATS else None
    scale = bias = ident = None
    if layout == SEAM:
        scale, bias, ident = extra
    rc, used, var = lib.gemm_run(av, bv, M, N, K, layout, out.origin, a_mn=a_mn, a_pitch=ap, b_mn=b_mn, b_pitch=bp,
                                 row_stride=out.row_stride, img_stride=out.img_stride, split_stride=out.split_stride, hw=hw,
                                 identity=ident, scale=scale, bias=bias, stats=None if st is None else st.origin, splits=splits,
                                 share=share, pair_fallback=fallback, sm_reserve=sm_reserve)
    torch.cuda.synchronize()
    assert rc == 0, lib.load().b200seg_last_error()
    assert used == want_splits, (used, want_splits)
    r = Run()
    r.variant, r.A, r.B, r.extra, r.per = var, A, B, extra, per
    if check_policy:
        want = policy(layout, M, N, K, splits, a_mn, b_mn, share, fallback, sw, lib.device_sms())
        assert VARIANTS[var] == want, (VARIANTS[var], want)
    r.d = out.values()
    r.splits = out.idx.shape[0]
    # fp64 reference, one slab per split (the k-blocks launch() assigns to it)
    Ad, Bd = A.double(), B.double()
    kps = per * 64
    r.slabs = [Ad[:, z * kps:(z + 1) * kps] @ Bd[:, z * kps:(z + 1) * kps].t() for z in range(r.splits)]
    r.ref = sum(r.slabs)
    if st is not None:
        r.mean, r.m2 = st.values()
    return r


def check_exact(r, layout, M, hw=0):
    if layout == SEAM:
        scale, bias, ident = r.extra
        want = seam_reference(r.ref, scale, bias, ident, M, hw).to(torch.bfloat16)
        bad = int((r.d[0] != want).sum())
        assert bad == 0, f"{bad} seam outputs differ from bf16_rn(relu(acc * scale + bias + identity))"
        return
    for z in range(r.splits):
        want = r.slabs[z].to(torch.bfloat16) if layout == BF16 else r.slabs[z]
        bad = int((r.d[z].double() != want.double()).sum())
        assert bad == 0, f"split {z}: {bad} of {want.numel()} elements differ from the exact reference"
    if layout == STATS:
        check_stats(r, M)


# about 4x the worst measured on a B200 (1000 W): 8.4e-8 for the mean, 1.8e-7 for M2
STATS_MEAN_TOL = 4e-7          # |mean - fp64 mean| / rms of the group
STATS_M2_TOL = 8e-7            # |M2 - fp64 M2| / sum v^2 of the group


def check_stats(r, M):
    mean, m2, sq, cnt = group_stats(r.d[0].double(), M)
    rms = (sq / cnt).sqrt().clamp_min(1e-30)
    em = ((r.mean - mean).abs() / rms).max().item()
    e2 = ((r.m2 - m2).abs() / sq.clamp_min(1e-30)).max().item()
    WORST["stats mean"] = max(WORST.get("stats mean", 0.0), em)
    WORST["stats M2"] = max(WORST.get("stats M2", 0.0), e2)
    assert em <= STATS_MEAN_TOL and e2 <= STATS_M2_TOL, (em, e2)
    return em, e2


WORST = {}


def check_accuracy(r, layout, tau=TAU):
    """|D - ref| <= tau * sum_k |a_ik b_kj| for every element (split slabs summed in fp64); records the worst ratio."""
    d = r.d.double().sum(0) if layout != BF16 else r.d[0].double()
    mag = r.A.double().abs() @ r.B.double().abs().t()
    ratio = ((d - r.ref).abs() / mag.clamp_min(1e-300)).max().item()
    WORST[LAYOUT_NAMES[layout]] = max(WORST.get(LAYOUT_NAMES[layout], 0.0), ratio)
    assert ratio <= tau, f"worst |D - ref| / sum|a b| = {ratio:.3g} > {tau:.3g}"
    return ratio


VARIANTS = []


@pytest.fixture(scope="module", autouse=True)
def _variant_table(lib):
    VARIANTS[:] = lib.gemm_variants()
    yield
    if WORST:
        print("\nworst error ratios (accuracy tier |D - ref| / sum|a b| per layout; statistics against fp64):",
              {k: f"{v:.3g}" for k, v in sorted(WORST.items())})


# ------------------------------------------------------------------ the exact tier under every switch setting
# (M, N, K, splits, a_mn, b_mn, hw, requested share): ragged M (1, 31, 100, 128, 129, 257 = half-empty pair, 384, 640), N ragged
# against 256 / 224 / 192, K below one k-block / one / ragged / many k-blocks, splits above the k-block count and uneven last splits
GENERIC = [
    (1, 77, 64, 1, False, False, 0, NONE),
    (31, 300, 8, 1, False, False, 0, SB),
    (100, 460, 72, 4, True, False, 0, SA),             # 2 k-blocks: splits clamp to 2
    (128, 200, 2056, 3, False, True, 0, PAIR),         # 33 k-blocks -> 3 splits of 11
    (129, 1000, 64, 1, False, False, 0, PAIR),
    (257, 520, 200, 3, True, True, 0, SB),             # 3 M-tiles (half-empty pair), 4 k-blocks -> 2 splits
    (384, 520, 5000, 3, False, False, 0, SA),          # 3 N-tiles (half-empty SHARE_A pair), 79 k-blocks -> 27 + 27 + 25
    (640, 777, 5000, 8, True, True, 0, PAIR),          # 79 k-blocks -> 7 x 10 + 9
    (640, 300, 2056, 1, False, False, 0, SA),
    (257, 1000, 72, 1, False, False, 0, NONE),
]
CASES = {
    F32: GENERIC,
    COLS: [
        (1, 77, 64, 1, False, False, 7, NONE),
        (100, 460, 72, 4, False, False, 33, SB),
        (128, 520, 200, 3, True, False, 129, SA),
        (257, 1000, 2056, 1, False, True, 250, PAIR),
        (640, 777, 5000, 3, False, False, 256, PAIR),
        (129, 300, 64, 1, True, True, 1, SB),
        (31, 4100, 64, 1, False, False, 4096, SA),
        (384, 520, 8, 1, False, False, 12, NONE),
    ],
    BF16: [
        (1, 8, 64, 1, False, False, 0, NONE),
        (31, 200, 72, 4, True, False, 0, SB),
        (129, 456, 2056, 3, False, True, 0, SA),
        (257, 520, 200, 2, False, False, 0, PAIR),
        (640, 1000, 5000, 8, True, True, 0, PAIR),
        (100, 520, 8, 1, False, False, 0, SA),
        (384, 776, 64, 1, False, False, 0, SB),
    ],
    # rows layouts: N from the register-store kernel's last-tile edges (8, 64, 136, 264, 320 = 64 left, 384 = 128 left, 392, 640);
    # hw 1, 31, 33, 127, 129, 4096 with several images, and the single-plane form (M <= hw, img_stride 0) as a negative hw below
    ROWS: [
        (100, 8, 64, 1, False, False, 1, PAIR),
        (279, 64, 72, 1, True, False, 31, PAIR),
        (132, 136, 8, 1, False, False, 33, PAIR),
        (381, 264, 2056, 1, True, False, 127, PAIR),
        (645, 320, 200, 1, False, False, 129, PAIR),
        (8192, 384, 64, 1, True, False, 4096, PAIR),
        (100, 392, 640, 1, False, False, -4096, PAIR),
        (1, 640, 72, 1, False, False, -31, PAIR),
        (129, 640, 5000, 1, False, False, -200, SB),
        (257, 392, 64, 1, False, False, 257, NONE),
        (640, 200, 64, 1, False, True, 128, PAIR),
        (384, 1000, 72, 1, False, False, 96, SA),
    ],
    STATS: [
        (132, 136, 64, 1, False, False, 33, PAIR),         # hw % 32 != 0: lane groups straddle images
        (279, 264, 72, 1, False, False, 31, NONE),
        (20, 64, 8, 1, False, False, -50, PAIR),           # M < 32, one M-tile: the forced pair
        (100, 320, 2056, 1, False, False, 100, PAIR),      # one M-tile, last group of 4 rows
        (257, 384, 200, 1, False, False, 257, PAIR),
        (645, 640, 640, 1, False, False, 129, PAIR),
        (1, 8, 64, 1, False, False, 1, PAIR),
    ],
    SEAM: [
        (1, 8, 64, 1, False, False, 1, PAIR),
        (100, 64, 72, 1, False, False, 100, PAIR),         # one M-tile: the pair is dropped
        (128, 256, 64, 1, False, False, 128, PAIR),        # ops.seam_conv3_tail (1, 64, 256, 8, 16)
        (35, 2048, 512, 1, False, False, 35, PAIR),        # ops.seam_conv3_tail (1, 512, 2048, 5, 7)
        (189, 264, 200, 1, False, False, 63, PAIR),
        (257, 392, 8, 1, False, False, 257, PAIR),
        (640, 520, 5000, 1, False, False, 320, PAIR),
        (300, 200, 64, 1, False, False, -400, NONE),
    ],
}
SWITCHES = [dict(sharing=m, narrow=n, dgrad=1) for m in (0, 1, 3, 4, 5) for n in (1, 0)]


def _settings(layout):
    if layout != ROWS:
        return SWITCHES
    return SWITCHES + [dict(sw, dgrad=d) for sw in SWITCHES for d in (0, 2)]


def _id(sw):
    return f"share{sw['sharing']}-narrow{sw['narrow']}-dgrad{sw['dgrad']}"


def _run_list(lib, layout, cases, sw, salt=0, exact=True, **kw):
    runs = []
    for i, (M, N, K, splits, a_mn, b_mn, hw, share) in enumerate(cases):
        single = hw < 0
        hw = abs(hw)
        fallback = PAIR if layout == SEAM else (SA if i % 2 else SB)
        r = run_case(lib, layout, M, N, K, splits=splits, a_mn=a_mn, b_mn=b_mn, hw=hw, share=share, fallback=fallback, sw=sw,
                     exact=exact, seed=1000 * layout + 10 * i + salt, off4=bool(i % 2) and layout in (F32, COLS),
                     single_plane=single, **kw)
        if exact:
            check_exact(r, layout, M, hw)
        runs.append(r)
    return runs


@pytest.mark.parametrize("layout,sw", [(lay, sw) for lay in (F32, COLS, BF16, ROWS, STATS, SEAM) for sw in _settings(lay)],
                         ids=lambda v: LAYOUT_NAMES[v] if isinstance(v, int) else _id(v))
def test_exact_tier_every_layout_and_switch(lib, layout, sw):
    set_switches(lib, **sw)
    _run_list(lib, layout, CASES[layout], dict(LOAD_TIME, **sw))


# ------------------------------------------------------------------ bench-sized problems, small grid
BENCH = [
    (F32, 640, 2048, 16770, 8, True, True, 0, PAIR, SA),          # the head's weight gradient (2 x 65 x 129 pixels), split-K
    (COLS, 2048, 16770, 640, 1, False, True, 8385, SB, SB),       # the head's data gradient, channels along M (dgrad mode 0)
    (ROWS, 65536, 2048, 640, 1, True, False, 4096, PAIR, SB),     # a pixel-major data gradient
    (BF16, 16770, 2048, 640, 1, True, False, 0, PAIR, SB),        # the seam-format data gradient
    (SEAM, 16770, 2048, 512, 1, False, False, 8385, PAIR, PAIR),  # the fused conv3 forward
    (STATS, 16770, 2048, 512, 1, False, False, 8385, PAIR, PAIR), # conv3 under batch statistics
]


@pytest.mark.parametrize("case", BENCH, ids=lambda c: LAYOUT_NAMES[c[0]])
def test_exact_tier_bench_sized(lib, case):
    layout, M, N, K, splits, a_mn, b_mn, hw, share, fallback = case
    sw = set_switches(lib, sharing=1, narrow=1, dgrad=1, fwd=1)
    r = run_case(lib, layout, M, N, K, splits=splits, a_mn=a_mn, b_mn=b_mn, hw=hw, share=share, fallback=fallback, sw=sw, seed=7)
    check_exact(r, layout, M, hw)


SMALL_GRID = [                            # about 40 work units on a grid of 2 CTAs (one pair): the rings wrap hundreds of times
    (F32, 640, 2048, 640, 1, False, False, 0, NONE),
    (F32, 1024, 2560, 640, 1, True, True, 0, PAIR),
    (COLS, 1024, 2560, 320, 1, False, True, 160, SB),
    (BF16, 640, 4096, 320, 2, False, False, 0, SA),
    (ROWS, 1024, 2560, 640, 1, False, False, 256, PAIR),
    (SEAM, 1024, 2560, 320, 1, False, False, 512, PAIR),
    (STATS, 1056, 2560, 320, 1, False, False, 33, PAIR),
]


@pytest.mark.parametrize("case", SMALL_GRID, ids=lambda c: f"{LAYOUT_NAMES[c[0]]}-{c[8]}")
def test_exact_tier_small_grid(lib, case):
    layout, M, N, K, splits, a_mn, b_mn, hw, share = case
    sw = set_switches(lib, sharing=1, narrow=1, dgrad=1, fwd=1)
    sms = lib.device_sms()
    r = run_case(lib, layout, M, N, K, splits=splits, a_mn=a_mn, b_mn=b_mn, hw=hw, share=share, fallback=SB, sw=sw, seed=8,
                 sm_reserve=sms - 2)
    check_exact(r, layout, M, hw)


# ------------------------------------------------------------------ accuracy tier, cross-layout and cross-geometry identity
@pytest.mark.parametrize("layout", [F32, COLS, ROWS], ids=lambda v: LAYOUT_NAMES[v])
@pytest.mark.parametrize("sharing", [0, 1, 4, 5])
def test_accuracy_tier(lib, layout, sharing):
    sw = set_switches(lib, sharing=sharing, narrow=1, dgrad=1, fwd=1)
    for r in _run_list(lib, layout, CASES[layout], sw, salt=5, exact=False):
        check_accuracy(r, layout)


@pytest.mark.parametrize("sharing", [0, 1, 3, 4, 5])
def test_bf16_equals_cast_of_f32_and_stats_c_equals_rows(lib, sharing):
    """Within one geometry (narrow tiles off: the bf16 layout never takes them), random data: BF16 == bf16(F32) per split slab,
    and the c of F32_NCHW_ROWS_STATS == F32_NCHW_ROWS under the same register-store pair."""
    sw = set_switches(lib, sharing=sharing, narrow=0, dgrad=1, fwd=1)
    g = torch.Generator().manual_seed(77)
    for M, N, K, splits, a_mn, b_mn, _, share in CASES[BF16]:
        data = (random_values(M, K, g).cuda(), random_values(N, K, g).cuda(), None)
        kw = dict(splits=splits, a_mn=a_mn, b_mn=b_mn, share=share, fallback=SB, sw=sw, data=data)
        f = run_case(lib, F32, M, N, K, **kw)
        b = run_case(lib, BF16, M, N, K, **kw)
        assert VARIANTS[f.variant] == VARIANTS[b.variant]
        assert torch.equal(b.d.view(torch.int16), f.d.to(torch.bfloat16).view(torch.int16)), (M, N, K)
    for M, N, K, _, a_mn, b_mn, hw, share in CASES[STATS]:
        data = (random_values(M, K, g).cuda(), random_values(N, K, g).cuda(), None)
        single = hw < 0
        s = run_case(lib, STATS, M, N, K, hw=abs(hw), share=PAIR, sw=sw, data=data, single_plane=single)
        check_stats(s, M)
        rows = run_case(lib, ROWS, M, N, K, hw=abs(hw), share=PAIR, fallback=PAIR, sw=sw, data=data, single_plane=single)
        if VARIANTS[rows.variant]["share"] == PAIR:               # (mode 0 gives the rows layout one CTA per tile)
            assert torch.equal(s.d.view(torch.int32), rows.d.view(torch.int32)), (M, N, K, hw)


GEOMETRIES = [  # (sharing mode, narrow, requested share, a_mn, b_mn): 1-CTA, multicast-B / -A, cta_group::2, 224 / 192 tiles, MN-major
    (1, 0, NONE, False, False), (1, 0, SB, False, False), (1, 0, SA, False, False), (1, 0, PAIR, False, False),
    (1, 1, NONE, False, False), (1, 1, SA, False, False), (1, 0, PAIR, True, True), (1, 0, SB, True, False), (1, 0, SA, False, True),
]


@pytest.mark.parametrize("shape", [(300, 148 * 224, 2056), (257, 148 * 192 - 40, 640), (640, 777, 5000)], ids=str)
def test_cross_geometry_bit_identity(lib, shape):
    """The same fp32 result bit for bit whatever the sharing geometry (cta_group::1 / ::2, multicast), tile width (256 / 224 /
    192), operand majorness or epilogue (rows layout: register-store pair, generic pair, one CTA): every tile sums its k-blocks
    in the same order with the same MMA shape along K.  Measured to hold on a B200; test_gemm_switches relies on it."""
    M, N, K = shape
    g = torch.Generator().manual_seed(M + N)
    data = (random_values(M, K, g).cuda(), random_values(N, K, g).cuda(), None)
    results, seen = {}, set()
    for mode, narrow, share, a_mn, b_mn in GEOMETRIES:
        sw = set_switches(lib, sharing=mode, narrow=narrow, dgrad=1, fwd=1)
        r = run_case(lib, F32, M, N, K, a_mn=a_mn, b_mn=b_mn, share=share, sw=sw, data=data)
        v = VARIANTS[r.variant]
        seen.add((v["share"], v["bn"]))
        results[(v["share"], v["bn"], a_mn, b_mn)] = r.d[0].view(torch.int32)
    for dgrad in (1, 2):                                             # the rows layout: register-store pair, generic pair, 1-CTA
        for mode in (1, 0, 5):
            sw = set_switches(lib, sharing=mode, narrow=1, dgrad=dgrad, fwd=1)
            r = run_case(lib, ROWS, M, N, K, hw=M, share=PAIR, fallback=SB, sw=sw, data=data)
            v = VARIANTS[r.variant]
            results[("rows", mode, dgrad, v["share"], v["bn"], v["rs"])] = r.d[0].view(torch.int32)
    first_key = next(iter(results))
    first = results[first_key]
    differ = [k for k, t in results.items() if not torch.equal(t, first)]
    print(f"{shape}: {len(results)} geometries, tile widths {sorted({b for _, b in seen})}, differing from {first_key}: {differ}")
    assert not differ


# ------------------------------------------------------------------ kernel choice, coverage, rejections, determinism
def _variant_of(lib, layout, M, N, K, sw, **kw):
    set_switches(lib, **sw)
    r = run_case(lib, layout, M, N, K, sw=dict(LOAD_TIME, **sw), **kw)
    check_exact(r, layout, M, kw.get("hw", 0))
    return VARIANTS[r.variant]


def test_policy_switches_reach_the_kernel_choice(lib):
    """b200seg.h's semantics, stated directly (run_case also checks each launch against POLICY)."""
    d = dict(sharing=1, narrow=0, dgrad=1)
    assert _variant_of(lib, F32, 300, 600, 64, d, share=PAIR)["share"] == PAIR
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=0), share=PAIR)["share"] == NONE            # mode 0: one CTA
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=0), share=SB)["share"] == NONE
    assert _variant_of(lib, F32, 300, 600, 64, d, share=SB)["share"] == SB
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=3), share=SB)["share"] == PAIR               # mode 3: B -> pair
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=3), share=SA)["share"] == SA
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=4), share=SA)["share"] == PAIR               # mode 4: A, B -> pair
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=4), share=SB)["share"] == PAIR
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=5), share=PAIR, fallback=SA)["share"] == SA  # mode 5: fallback
    assert _variant_of(lib, F32, 300, 600, 64, dict(d, sharing=5), share=PAIR, fallback=SB)["share"] == SB
    v = _variant_of(lib, SEAM, 300, 64, 64, dict(d, sharing=5), share=PAIR, fallback=PAIR, hw=300)          # the seam GEMM keeps its pair
    assert v["share"] == PAIR and v["seam"]
    for mode in (0, 1, 5):                                                                                 # STATS: always a pair
        v = _variant_of(lib, STATS, 100, 64, 64, dict(d, sharing=mode), share=NONE, hw=100)
        assert v["share"] == PAIR and v["rs"] and v["stats"]
    assert _variant_of(lib, F32, 128, 600, 64, d, share=PAIR)["share"] == NONE                               # one M-tile: no pair
    assert _variant_of(lib, F32, 100, 600, 64, d, share=SB)["share"] == NONE
    assert _variant_of(lib, F32, 300, 256, 64, d, share=SA)["share"] == NONE                                 # one N-tile: no A pair
    assert _variant_of(lib, SEAM, 128, 64, 64, d, share=PAIR, fallback=PAIR, hw=128)["share"] == NONE
    # the rows layout takes the register-store kernel on pairs, except under dgrad mode 2 (streaming stores, generic kernel)
    for dgrad, rs in ((0, 1), (1, 1), (2, 0)):
        v = _variant_of(lib, ROWS, 300, 64, 64, dict(d, dgrad=dgrad), share=PAIR, hw=300)
        assert v["share"] == PAIR and v["rs"] == rs
    assert not _variant_of(lib, ROWS, 300, 64, 64, dict(d, sharing=5), share=PAIR, hw=300)["rs"]
    # narrow tiles: 224 / 192 columns where they make whole rounds of the SMs, only with the switch on and K-major fp32 output
    sms = lib.device_sms()
    assert _variant_of(lib, F32, 100, sms * 224, 64, dict(d, narrow=1), share=NONE)["bn"] == 224
    assert _variant_of(lib, F32, 100, sms * 192, 64, dict(d, narrow=1), share=NONE)["bn"] == 192
    assert _variant_of(lib, F32, 100, sms * 224, 64, d, share=NONE)["bn"] == 256
    assert _variant_of(lib, ROWS, 100, sms * 224, 64, dict(d, narrow=1, sharing=0), share=PAIR, hw=100)["bn"] == 224
    assert _variant_of(lib, BF16, 100, sms * 224, 64, dict(d, narrow=1), share=NONE)["bn"] == 256


def _coverage_cases(sms):
    """(layout, M, N, K, switches, kwargs): between them every kernel of the table."""
    off = dict(sharing=1, narrow=0, dgrad=1)
    on = dict(off, narrow=1)
    cases = []
    for a_mn in (False, True):
        for b_mn in (False, True):
            for share in (NONE, SB, SA, PAIR):
                cases.append((F32, 300, 600, 200, off, dict(a_mn=a_mn, b_mn=b_mn, share=share, splits=2)))
    for share in (NONE, SA):
        cases.append((F32, 100, sms * 224, 64, on, dict(share=share)))
        cases.append((COLS, 100, sms * 192, 64, on, dict(share=share, hw=4096)))
    for a_mn in (False, True):
        cases.append((ROWS, 300, 320, 200, off, dict(a_mn=a_mn, share=PAIR, hw=100)))
    cases.append((SEAM, 100, 136, 200, off, dict(share=PAIR, fallback=PAIR, hw=100)))
    cases.append((SEAM, 300, 136, 200, off, dict(share=PAIR, fallback=PAIR, hw=100)))
    cases.append((STATS, 300, 136, 200, off, dict(share=PAIR, hw=100)))
    return cases


def test_every_kernel_launched_and_deterministic(lib):
    """A compact list of exact-tier cases launches every index of the variant table (a kernel added without a test fails here);
    each is also run twice on random data: bit-identical (no atomics; split slabs are separate)."""
    launched = set()
    for layout, M, N, K, sw, kw in _coverage_cases(lib.device_sms()):
        set_switches(lib, **sw)
        full = dict(LOAD_TIME, **sw)
        r = run_case(lib, layout, M, N, K, sw=full, seed=3, **kw)
        check_exact(r, layout, M, kw.get("hw", 0))
        launched.add(r.variant)
        g = torch.Generator().manual_seed(4)
        data = (random_values(M, K, g).cuda(), random_values(N, K, g).cuda(), r.extra)
        r1 = run_case(lib, layout, M, N, K, sw=full, data=data, **kw)
        r2 = run_case(lib, layout, M, N, K, sw=full, data=data, **kw)
        assert r1.variant == r2.variant == r.variant
        view = torch.int16 if layout in (BF16, SEAM) else torch.int32
        assert torch.equal(r1.d.view(view), r2.d.view(view)), (LAYOUT_NAMES[layout], VARIANTS[r.variant])
        if layout == STATS:
            assert torch.equal(r1.mean, r2.mean) and torch.equal(r1.m2, r2.m2)
    print(f"GEMM kernels launched: {len(launched)}/{len(VARIANTS)}")
    assert launched == set(range(len(VARIANTS))), sorted(set(range(len(VARIANTS))) - launched)


def _reject(lib, layout, M, N, K, *, a_off=0, a_pitch_extra=0, out_off=0, **kw):
    """A launch with one bad argument: B200SEG_ERR_ARG, variant -1 for the layout checks, output and stats untouched."""
    set_switches(lib, sharing=1, narrow=1, dgrad=1, fwd=1)
    g = torch.Generator().manual_seed(5)
    A, B = exact_values(M, K, g).cuda(), exact_values(N, K, g).cuda()
    a_mn, b_mn = kw.pop("a_mn", False), kw.pop("b_mn", False)
    av, ap = operand(A, a_mn)
    if a_off or a_pitch_extra:                                         # re-seat A: misaligned base or a pitch not a multiple of 8
        ap = av.shape[1] + a_pitch_extra
        buf = torch.zeros(a_off + av.shape[0] * ap + 64, dtype=torch.bfloat16, device="cuda")
        av = buf[a_off:a_off + av.shape[0] * ap].view(av.shape[0], ap)[:, :av.shape[1]]
        av.copy_((A.t() if a_mn else A).to(torch.bfloat16))
    bv, bp = operand(B, b_mn)
    bf16 = layout in (BF16, SEAM)
    out = torch.full((GUARD + M * N * 4 + 8 * N + GUARD,), BF16_SENTINEL if bf16 else F32_SENTINEL,
                     dtype=torch.int16 if bf16 else torch.int32, device="cuda")
    before = out.clone()
    stats = torch.full((2 * (cdiv(M, 32) * N + 16),), F32_SENTINEL, dtype=torch.int32, device="cuda")
    seam = {}
    if layout == SEAM:
        seam = dict(zip(("scale", "bias", "identity"), seam_inputs(M, N, kw["hw"], g)))
    origin = out[GUARD + out_off:].view(torch.bfloat16 if bf16 else torch.float32)
    rc, _, var = lib.gemm_run(av, bv, M, N, K, layout, origin, a_mn=a_mn, a_pitch=ap, b_mn=b_mn, b_pitch=bp,
                              stats=stats.view(torch.float32) if layout == STATS else None, check=False, **seam, **kw)
    torch.cuda.synchronize()
    assert rc == ERR_ARG, rc
    assert torch.equal(out, before) and bool((stats == F32_SENTINEL).all())
    return var


def test_rejections_leave_the_output_untouched(lib):
    assert _reject(lib, SEAM, 256, 64, 64, hw=256, a_mn=True) == -1                 # SEAM / STATS: K-major operands only
    assert _reject(lib, SEAM, 256, 64, 64, hw=256, b_mn=True) == -1
    assert _reject(lib, STATS, 256, 64, 64, hw=256, a_mn=True) == -1
    assert _reject(lib, STATS, 256, 64, 64, hw=256, b_mn=True) == -1
    assert _reject(lib, STATS, 256, 64, 640, hw=256, splits=2) == -1                # no split-K for the rows layouts
    assert _reject(lib, ROWS, 256, 64, 640, hw=256, splits=2, img_stride=64 * 256) == -1
    assert _reject(lib, SEAM, 256, 64, 640, hw=256, splits=2) == -1
    assert _reject(lib, BF16, 64, 12, 64, row_stride=16) == -1                      # bf16: N % 8, row pitch % 8, 16-byte base
    assert _reject(lib, BF16, 64, 16, 64, row_stride=20) == -1
    assert _reject(lib, BF16, 64, 16, 64, row_stride=16, out_off=1) == -1
    assert _reject(lib, SEAM, 64, 12, 64, hw=64) == -1
    assert _reject(lib, SEAM, 64, 16, 64, hw=64, out_off=1) == -1
    assert _reject(lib, ROWS, 100, 64, 64, hw=33, img_stride=64 * 33) == -1         # M > hw and M % hw != 0
    assert _reject(lib, STATS, 100, 64, 64, hw=33, img_stride=64 * 33) == -1
    assert _reject(lib, COLS, 64, 64, 64, hw=0, row_stride=64) == -1                # the column map needs hw > 0
    assert _reject(lib, F32, 64, 64, 64, row_stride=64, share=3) == -1              # not a sharing geometry
    assert _reject(lib, F32, 64, 64, 64, row_stride=64, a_off=1) == -1                # operand base not 16-byte aligned
    assert _reject(lib, F32, 64, 64, 64, row_stride=64, a_pitch_extra=4) == -1        # operand pitch not a multiple of 8
    assert _reject(lib, F32, 64, 64, 64, row_stride=64, a_mn=True, a_pitch_extra=4) == -1
