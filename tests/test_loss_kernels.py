"""The loss kernels against an fp64 reference of the same operation, at the shapes, label values and logit ranges where they
can go wrong:

  K2  fused align-corners upsample + softmax cross-entropy (ignore_index) and its gradient: the CTA-tile kernel
      (csrc/ce_kernels.cu) and the warp-tile kernel (csrc/ce_v2_kernels.cu), the fp32 NCHW and the packed bf16 backward;
  K5  the FADA soft-label tail: upsample + q = min(softmax(seg / T), clamp) + soft-label CE (csrc/ce_kernels.cu);
  K3  soft-label CE on materialised operands, vectorised and scalar paths (csrc/softce_kernels.cu).

The reference is built from the same fp32 interpolation taps the kernels and ATen use (scale = f32(in-1) / f32(out-1),
src = f32(scale * dst), i0 = int(src), i1 = min(i0 + 1, in - 1), l1 = src - i0, l0 = 1 - l1) as dense fp64 matrices Ry [H, h],
Rx [W, w]: the upsample is Ry x Rx^T per plane and its adjoint Ry^T G Rx.  Everything after the taps is fp64.

Bars follow from fp32 arithmetic, not from one flat tolerance: an fp32 kernel is off by a few units of 2^-24 of the magnitudes
it handles, so each check is |got - ref| <= k * 2^-24 * (a magnitude of the same operation), with k calibrated on a B200.
The dispatch (which kernel instantiation runs for which shape) is mirrored here; a CPU test asserts that the case tables reach
every branch of it, a GPU test that the mirror names the kernel that actually runs."""
import math
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu
EPS = 2.0 ** -24

# k of each bar: about 4x the worst ratio |got - ref| / (2^-24 * magnitude) measured on a B200 (1000 W) over this file's cases,
# which was: K2 loss 0.96, K2 gradient 2.61, K2 bias 1.34, K5 loss 0.24, K5 gradient 1.01, K3 loss 1.79, K3 gradient 3.3
K2_LOSS_K = 4.0
K2_GRAD_K = 12.0
K2_BIAS_K = 6.0
K5_LOSS_K = 1.0
K5_GRAD_K = 4.0
K3_LOSS_K = 8.0
K3_GRAD_K = 14.0
# smallest normal fp32: the kernels' exponentials (ex2.approx.ftz) flush anything below it to 0
TINY = 2.0 ** -126

WORST = {}


def _record(name, err, unit):
    """err / unit where unit > 0 (entries whose magnitude is 0 must match exactly); records the worst ratio per check."""
    err = err.double().cpu()
    unit = unit.double().cpu()
    exact = unit == 0
    assert not (exact & (err != 0)).any(), f"{name}: {int((exact & (err != 0)).sum())} entries of zero magnitude are not exact"
    ratio = (err[~exact] / unit[~exact]).max().item() if (~exact).any() else 0.0
    WORST[name] = max(WORST.get(name, 0.0), ratio)
    return ratio


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if WORST:
        print("\nworst |got - ref| / (2^-24 * magnitude):", {k: round(v, 2) for k, v in sorted(WORST.items())})


# ============================================================================================================ fp64 reference
def ac_taps(n_in, n_out):
    """fp32 align-corners taps (common.cuh ac_scale / ac_tap == ATen's area_pixel_compute_scale + source index for float)."""
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0.0)
    src = (np.float32(scale) * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = src.astype(np.int64)
    i1 = np.minimum(i0 + 1, n_in - 1)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1.0) - l1).astype(np.float32)
    return i0, i1, l0, l1


def interp_matrix(n_in, n_out):
    """fp64 [n_out, n_in]: row d holds l0 at i0(d) and l1 at i1(d) (summed where they coincide)."""
    i0, i1, l0, l1 = ac_taps(n_in, n_out)
    R = np.zeros((n_out, n_in))
    np.add.at(R, (np.arange(n_out), i0), l0.astype(np.float64))
    np.add.at(R, (np.arange(n_out), i1), l1.astype(np.float64))
    return torch.from_numpy(R)


def incidence(n_in, n_out):
    """bool [n_out, n_in]: output d reads source i (either tap, whatever its weight)."""
    i0, i1, _, _ = ac_taps(n_in, n_out)
    M = np.zeros((n_out, n_in), dtype=bool)
    M[np.arange(n_out), i0] = True
    M[np.arange(n_out), i1] = True
    return torch.from_numpy(M)


def up(x, Ry, Rx):
    return torch.einsum("Hh,nchw,Ww->ncHW", Ry, x, Rx)


def adj(G, Ry, Rx):
    return torch.einsum("Hh,ncHW,Ww->nchw", Ry, G, Rx)


def k2_reference(x, labels, ignore_index, T):
    """fp64 CrossEntropyLoss(ignore_index)(interpolate(x) / T, labels) with labels outside [0, C) excluded like ignore_index.
    Returns loss, d loss / d x, n_valid, the bar magnitudes S (loss) and A (per gradient element), and the most each gradient
    element can lose to exponentials below the fp32 normal range, which the kernels flush to 0: U for the CTA-tile kernel
    (exponentials relative to the pixel's maximum: a softmax entry below 2^-126 is lost), U2 for the warp-tile kernel (relative
    to M, the maximum over both source rows of the pixel's column: an entry below 2^-126 * exp(M - lse) is lost, unless that
    factor exceeds 1e30, where the kernel takes its exact path with the pixel's own maximum)."""
    x = x.detach().double().cpu()
    lab = labels.detach().cpu().long()
    N, C, h, w = x.shape
    H, W = lab.shape[-2:]
    Ry, Rx = interp_matrix(h, H), interp_matrix(w, W)
    z = up(x, Ry, Rx) / T
    valid = (lab >= 0) & (lab < C) & (lab != ignore_index)
    n_valid = int(valid.sum())
    idx = torch.where(valid, lab, torch.zeros_like(lab))
    lse = torch.logsumexp(z, 1)
    zl = z.gather(1, idx[:, None])[:, 0]
    vf = valid.double()
    loss = ((lse - zl) * vf).sum() / n_valid if n_valid else torch.tensor(float("nan"), dtype=torch.float64)
    sm = torch.softmax(z, 1)
    oh = F.one_hot(idx, C).permute(0, 3, 1, 2).double() * vf[:, None]
    denom = max(n_valid, 1) * T
    grad = adj((sm - oh) * vf[:, None], Ry, Rx) / denom
    zmax = z.amax(1)
    S = ((zmax.abs() + lse.abs() + zl.abs()) * vf).sum() / max(n_valid, 1)
    A = adj((sm + oh) * (vf * (1 + z.abs().amax(1)))[:, None], Ry, Rx) / denom
    U = adj(TINY * vf[:, None].expand_as(z), Ry, Rx) / denom
    hx = torch.einsum("nchw,Ww->nchW", x, Rx).amax(1) / T                 # per source row and output column, max over classes
    i0, i1, _, _ = ac_taps(h, H)
    M = torch.maximum(hx[:, torch.from_numpy(i0)], hx[:, torch.from_numpy(i1)])
    lift = torch.where(M - lse < math.log(1e30), torch.exp(M - lse), torch.ones_like(lse))
    U2 = adj(TINY * (vf * lift)[:, None].expand_as(z), Ry, Rx) / denom
    return loss, grad, n_valid, S, A, U, U2


def soft_ce_reference(pred, soft, wts):
    """fp64 mean_{N,H,W}( [w *] sum_c -q_c log_softmax(p)_c ) and its gradient, with shift-invariant bar magnitudes: they are
    made of logit differences p - max p, so a logit offset common to all classes changes neither the result nor the bar."""
    p = pred.detach().double().cpu()
    q = soft.detach().double().cpu()
    N, K, H, W = p.shape
    w = torch.ones(N, H, W, dtype=torch.float64) if wts is None else wts.detach().double().cpu().reshape(N, H, W)
    m = p.amax(1, keepdim=True)
    lse = torch.logsumexp(p, 1, keepdim=True)
    sq = q.sum(1, keepdim=True)
    px = (q * (lse - p)).sum(1) * w
    cnt = N * H * W
    loss = px.sum() / cnt
    sm = torch.softmax(p, 1)
    grad = (sm * sq - q) * w[:, None] / cnt
    d = (p - m).abs()
    S = (w.abs() * (q.abs().sum(1) * (1 + (lse - m)[:, 0].abs()) + (q.abs() * d).sum(1))).sum() / cnt
    A = (sm * q.abs().sum(1, keepdim=True) * (1 + d.amax(1, keepdim=True)) + q.abs()) * w.abs()[:, None] / cnt
    return loss, grad, S, A


def k5_reference(d, seg, size, slot, T, clamp):
    """fp64 soft-label CE of interpolate(d) against q = min(softmax(interpolate(seg) / T), clamp) in channel slot `slot`, its
    gradient w.r.t. d, and bar magnitudes.  q is built in fp32 by the kernel from fp32-interpolated logits: its error scales
    with max |seg / T|, which is folded into both magnitudes."""
    dd = d.detach().double().cpu()
    ss = seg.detach().double().cpu()
    N, K, h, w = dd.shape
    C = K // 2
    H, W = size
    Ry, Rx = interp_matrix(h, H), interp_matrix(w, W)
    D = up(dd, Ry, Rx)
    Sg = up(ss, Ry, Rx) / T
    qc = torch.softmax(Sg, 1).clamp(max=clamp)
    Q = torch.zeros_like(D)
    Q[:, slot * C:(slot + 1) * C] = qc
    lse = torch.logsumexp(D, 1, keepdim=True)
    sq = Q.sum(1, keepdim=True)
    cnt = N * H * W
    loss = (Q * (lse - D)).sum(1).sum() / cnt
    smD = torch.softmax(D, 1)
    grad = adj(smD * sq - Q, Ry, Rx) / cnt
    seg_mag = 1 + Sg.abs().amax(1)
    S = (((sq[:, 0] * (D.amax(1).abs() + lse[:, 0].abs()) + (Q * D.abs()).sum(1))) * seg_mag).sum() / cnt
    A = adj((smD * sq + Q) * ((1 + D.abs().amax(1)) * seg_mag)[:, None], Ry, Rx) / cnt
    return loss, grad, S, A


# ============================================================================================ dispatch mirror (host side)
def _v2_eligible(N, C, h, w, H, W):
    """ce_v2_kernels.cu k2v2_eligible."""
    if C not in (19, 2) or H < h or W < w or H < 2 or W < 2:
        return False
    i0, i1, _, _ = ac_taps(w, W)
    for xa in range(0, W, 32):
        xb = min(xa + 32, W) - 1
        lo, hi = int(i0[xa]), int(i0[xb])
        hi += 1 if hi < w - 1 else 0
        if hi - lo + 1 > 8:
            return False
    return True


def k2_dispatch(variant, N, C, h, w, H, W, u8, w_aligned=True):
    """The K2 main kernel k2_forward (ce_kernels.cu) picks: ("v2", CT, LM) for the warp-tile kernel with label mode LM
    (0 int64, 1 uint8 4-byte aligned rows, 2 uint8 otherwise) or ("cta", CT) for the CTA-tile kernel."""
    if variant != 0 and (C == 19 or variant == 2) and _v2_eligible(N, C, h, w, H, W):
        return ("v2", C, (1 if (W % 4 == 0 and w_aligned) else 2) if u8 else 0)
    return ("cta", 2 if C == 2 else 19 if C == 19 else 8 if C <= 8 else 32)


def k2_row_paths(w, W):
    """Row-load paths the CTA-tile kernel's warps take: 'staged' when a warp's 32 columns read < 8 source columns, else
    'global' (k2_row_load)."""
    i0, i1, _, _ = ac_taps(w, W)
    paths = set()
    for x0 in range(0, ((W + 127) // 128) * 128, 32):
        lo, hi = int(i0[min(x0, W - 1)]), int(i1[min(x0 + 31, W - 1)])
        paths.add("staged" if hi - lo < 8 else "global")
    return paths


def k5_dispatch(C, slot):
    return (19 if C == 19 else 2 if C == 2 else 8 if C <= 8 else 16 if C <= 16 else 24 if C <= 24 else 32, slot)


def k3_dispatch(K, vec, stats):
    """(forward kernel, backward kernel) k3_forward / k3_backward (softce_kernels.cu) launch."""
    kt = 4 if K <= 4 else 38 if K <= 38 else 64
    fwd = "fwd_v4" if vec else f"fwd<{kt}>"
    bwd = "bwd_stats_v4" if (vec and stats) else f"bwd<{kt}>"
    return fwd, bwd


# ============================================================================================================ case tables
# (N, C, h, w, H, W, label dtype, ignore_index, label recipe, logit recipe, T)
#   label recipe: "plain" (10 % ignore_index), "oob" (plus labels >= C and, for int64, negative ones), "hole" (a whole
#   CTA tile without a valid label inside a valid frame), "frame" (frame 1 all ignore_index), "none" (all ignore_index)
#   logit recipe: "n2" 2 * randn, "s60" 60 * randn (neighbouring source pixels far apart), "o1000" randn + 1000
I64, U8 = "int64", "uint8"
K2_CASES = [
    # class counts, both kernels where the warp-tile kernel is eligible (C = 2, 19)
    *[(2, C, 9, 13, 50, 70, I64, 255, "plain", "n2", 1.0) for C in (1, 2, 3, 8, 9, 19, 20, 31, 32)],
    (2, 19, 9, 13, 50, 70, U8, 255, "plain", "n2", 1.8),
    (2, 2, 9, 13, 50, 68, U8, 255, "plain", "n2", 1.8),
    # geometry
    (1, 19, 16, 40, 16, 40, I64, 255, "plain", "n2", 1.0),          # identity: unstaged (global-load) rows
    (1, 8, 16, 40, 16, 40, I64, 255, "plain", "n2", 1.0),
    (1, 32, 12, 30, 12, 30, I64, 255, "plain", "n2", 1.0),
    (1, 2, 12, 30, 12, 30, U8, 255, "plain", "n2", 1.0),
    (1, 19, 20, 30, 30, 45, I64, 255, "plain", "n2", 1.0),          # 1.5x
    (2, 19, 9, 17, 33, 65, I64, 255, "plain", "n2", 1.8),           # 4x
    (1, 19, 8, 16, 57, 121, I64, 255, "plain", "n2", 1.0),          # 8x
    (1, 19, 2, 5, 1024, 37, I64, 255, "plain", "n2", 1.0),          # 2-row source to 1024 rows
    (1, 19, 1, 7, 5, 50, I64, 255, "plain", "n2", 1.0),             # h = 1
    (1, 19, 7, 1, 50, 5, I64, 255, "plain", "n2", 1.0),             # w = 1
    (1, 19, 4, 6, 1, 40, I64, 255, "plain", "n2", 1.0),             # H = 1
    (1, 19, 6, 4, 40, 1, I64, 255, "plain", "n2", 1.0),             # W = 1
    (2, 19, 5, 6, 37, 20, U8, 255, "plain", "n2", 1.0),             # W < 32
    (2, 19, 13, 29, 97, 203, I64, 255, "plain", "n2", 1.0),         # H, W not multiples of 32 / 128
    (2, 2, 13, 29, 97, 203, U8, 255, "plain", "n2", 1.0),
    (1, 19, 8, 8, 40, 32, I64, 255, "plain", "n2", 1.0),            # warp tile spans exactly 8 source columns: eligible
    (1, 19, 9, 9, 40, 32, I64, 255, "plain", "n2", 1.0),            # 9: falls back to the CTA-tile kernel
    (3, 19, 9, 17, 64, 128, I64, 255, "plain", "n2", 1.0),          # N > 1, tiles ending at the frame edge
    (3, 2, 9, 17, 70, 150, I64, 255, "plain", "n2", 1.0),
    # labels
    (2, 19, 9, 13, 50, 70, I64, 0, "plain", "n2", 1.0),             # ignore_index 0
    (2, 8, 9, 13, 50, 70, I64, -100, "oob", "n2", 1.0),             # -100, labels >= C and negative labels
    (2, 19, 9, 13, 50, 70, U8, -100, "oob", "n2", 1.0),
    (2, 19, 9, 13, 50, 70, I64, 19, "oob", "n2", 1.0),              # ignore_index == C
    (2, 2, 9, 13, 50, 70, U8, 7, "oob", "n2", 1.0),                 # ignore_index > C
    (1, 32, 9, 13, 50, 70, U8, 255, "oob", "n2", 1.0),
    (1, 19, 13, 37, 96, 300, I64, 255, "hole", "n2", 1.0),          # a tile with no valid label inside a valid frame
    (1, 2, 13, 37, 96, 300, U8, 255, "hole", "n2", 1.0),
    (3, 19, 9, 17, 64, 96, I64, 255, "frame", "n2", 1.0),           # an all-ignored frame among valid ones
    (3, 9, 9, 17, 64, 96, U8, 255, "frame", "n2", 1.0),
    # logits
    (2, 19, 9, 13, 50, 70, I64, 255, "plain", "s60", 1.0),
    (2, 2, 9, 13, 50, 70, I64, 255, "plain", "s60", 1.8),
    (1, 9, 9, 13, 50, 70, U8, 255, "plain", "s60", 1.0),
    (2, 19, 9, 13, 50, 70, I64, 255, "plain", "o1000", 1.0),
    (1, 3, 9, 13, 50, 70, I64, 255, "plain", "o1000", 1.8),
]

# (N, C, h, w, H, W, slot, clamp, T)
K5_CASES = [
    *[(2, C, 7, 9, 33, 47, slot, (0.9, 1.0, 0.05)[(C + slot) % 3], (1.8, 1.0)[slot]) for C in (1, 2, 3, 8, 9, 16, 19, 24, 32)
      for slot in (0, 1)],
    (1, 19, 1, 5, 9, 40, 1, 0.9, 1.8),                               # h = 1
    (1, 19, 12, 12, 12, 12, 0, 0.9, 1.8),                            # identity
    (2, 2, 5, 6, 37, 20, 1, 0.9, 1.8),                               # W < 32
    (1, 19, 13, 29, 97, 203, 0, 0.9, 1.8),                           # several tiles, ragged edges
]

# (N, K, H, W, layout, weighted, soft recipe, offset); layout: "vec" (H*W % 4 == 0, aligned), "odd" (odd H*W),
# "off4" (H*W % 4 == 0, a view 4 bytes into its buffer); soft recipe: "dense", "zero_rows" (some pixels' q all 0),
# "zero_w" (some pixel weights 0)
K3_CASES = [
    *[(2, K, 12, 20, "vec", K % 2 == 0, "dense", 0.0) for K in (1, 4, 5, 38, 39, 64)],
    *[(2, K, 9, 13, "odd", K % 2 == 1, "dense", 0.0) for K in (1, 4, 5, 38, 39, 64)],
    *[(1, K, 8, 12, "off4", True, "dense", 0.0) for K in (4, 38, 64)],
    (2, 38, 12, 20, "vec", True, "zero_rows", 0.0),
    (2, 38, 9, 13, "odd", False, "zero_rows", 0.0),
    (2, 38, 12, 20, "vec", True, "zero_w", 0.0),
    (2, 5, 9, 13, "odd", True, "zero_w", 0.0),
    (2, 38, 12, 20, "vec", False, "dense", 1000.0),                 # a common logit offset cancels in the loss
    (2, 38, 9, 13, "odd", True, "dense", 1000.0),
    (2, 64, 12, 20, "vec", True, "dense", 100.0),
    (1, 4, 8, 12, "off4", False, "dense", 1000.0),
]


def _case_id(c):
    return "-".join(str(v) for v in c)


# ================================================================================================================ inputs
def k2_inputs(case, seed):
    N, C, h, w, H, W, ldt, ign, lrec, xrec, T = case
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, C, h, w, generator=g)
    x = {"n2": 2.0 * x, "s60": 60.0 * x, "o1000": x + 1000.0}[xrec]
    lab = torch.randint(0, C, (N, H, W), generator=g)
    fill = 255 if ign < 0 and ldt == U8 else ign
    lab[torch.rand(N, H, W, generator=g) < 0.1] = fill
    if lrec == "oob":
        r = torch.rand(N, H, W, generator=g)
        lab[r < 0.05] = C
        lab[(r >= 0.05) & (r < 0.1)] = 200
        if ldt == I64:
            lab[(r >= 0.1) & (r < 0.15)] = -1
            lab[(r >= 0.15) & (r < 0.2)] = -7
    elif lrec == "hole":
        lab[0, 32:64, 128:256] = fill
    elif lrec == "frame":
        lab[1] = fill
    elif lrec == "none":
        lab[:] = fill
    return x.float(), lab.to(torch.uint8 if ldt == U8 else torch.int64), ign, T


# ================================================================================================== CPU: the reference itself
@pytest.mark.parametrize("N,C,h,w,H,W", [(2, 5, 4, 6, 9, 13), (1, 3, 1, 5, 4, 11), (1, 4, 5, 1, 12, 3), (1, 2, 3, 4, 1, 7),
                                         (1, 3, 4, 3, 6, 1), (1, 2, 7, 9, 7, 9), (1, 3, 9, 12, 4, 5)])
def test_reference_matches_torch_fp64(N, C, h, w, H, W):
    """The fp64 reference (dense tap matrices, analytic gradients) against F.interpolate(align_corners=True) + F.cross_entropy /
    log_softmax in fp64 with autograd, 1-row, 1-column and down-sampling shapes included.  ATen's fp64 taps are computed in fp64,
    the reference's in fp32 (as the kernels'), so the two agree to fp32 rounding of the tap weights."""
    g = torch.Generator().manual_seed(N + C + h + w + H + W)
    x = (2.0 * torch.randn(N, C, h, w, generator=g)).float()
    lab = torch.randint(0, C, (N, H, W), generator=g)
    lab[torch.rand(N, H, W, generator=g) < 0.2] = 255
    if lab.ne(255).sum() == 0:
        lab[0, 0, 0] = 0
    T = 1.8
    xd = x.double().requires_grad_(True)
    z = F.interpolate(xd, size=(H, W), mode="bilinear", align_corners=True)
    want = F.cross_entropy(z / T, lab, ignore_index=255)
    want_g, = torch.autograd.grad(want, xd)
    loss, grad, n_valid, S, A, _, _ = k2_reference(x, lab, 255, T)
    Ry, Rx = interp_matrix(h, H), interp_matrix(w, W)
    assert (up(x.double(), Ry, Rx) - z.detach()).abs().max() <= 1e-6 * (1 + x.abs().max())
    assert n_valid == int(lab.ne(255).sum())
    assert abs(loss - want.item()) <= 1e-6 * S
    assert ((grad - want_g).abs() <= 1e-6 * A + 1e-12).all()
    # soft-label CE and the K5 tail against log_softmax on materialised fp64 tensors
    d = torch.randn(N, 2 * C, h, w, generator=g).float()
    seg = (3.0 * torch.randn(N, C, h, w, generator=g)).float()
    for slot in (0, 1):
        dd = d.double().requires_grad_(True)
        D = F.interpolate(dd, size=(H, W), mode="bilinear", align_corners=True)
        q = torch.softmax(F.interpolate(seg.double(), size=(H, W), mode="bilinear", align_corners=True) / T, 1).clamp(max=0.9)
        Q = torch.cat((q, torch.zeros_like(q)) if slot == 0 else (torch.zeros_like(q), q), 1)
        want = (-Q * F.log_softmax(D, 1)).sum(1).mean()
        want_g, = torch.autograd.grad(want, dd)
        loss, grad, S, A = k5_reference(d, seg, (H, W), slot, T, 0.9)
        assert abs(loss - want.item()) <= 1e-6 * S
        assert ((grad - want_g).abs() <= 1e-6 * A + 1e-12).all()
    p = (3.0 * torch.randn(N, 2 * C, H, W, generator=g)).double().requires_grad_(True)
    soft = torch.softmax(torch.randn(N, 2 * C, H, W, generator=g), 1).double()
    wts = torch.rand(N, H, W, generator=g).double()
    want = ((-soft * F.log_softmax(p, 1)).sum(1) * wts).mean()
    want_g, = torch.autograd.grad(want, p)
    loss, grad, S, A = soft_ce_reference(p, soft, wts)
    assert abs(loss - want.item()) <= 1e-12 * S
    assert ((grad - want_g).abs() <= 1e-12 * A + 1e-15).all()


def test_reference_excludes_out_of_range_labels():
    """Labels >= C and negative labels count like ignore_index in the reference (the kernels' documented behaviour)."""
    x = torch.randn(1, 3, 4, 5).float()
    lab = torch.randint(0, 3, (1, 8, 9))
    lab[0, :2] = 3
    lab[0, 2, :] = -5
    keep = (lab >= 0) & (lab < 3)
    loss, _, n_valid, _, _, _, _ = k2_reference(x, lab, 255, 1.0)
    masked = torch.where(keep, lab, torch.full_like(lab, 255))
    want = F.cross_entropy(F.interpolate(x.double(), size=(8, 9), mode="bilinear", align_corners=True), masked, ignore_index=255)
    assert n_valid == int(keep.sum())
    assert abs(loss - want.item()) <= 1e-6


def test_case_tables_reach_every_dispatch_branch():
    """Every kernel instantiation and path the launchers can pick is reached by at least one case of the tables below."""
    k2 = set()
    for (N, C, h, w, H, W, ldt, *_rest) in K2_CASES:
        for variant in (0, 2):
            k2.add(k2_dispatch(variant, N, C, h, w, H, W, ldt == U8))
        if k2_dispatch(0, N, C, h, w, H, W, False)[0] == "cta":
            k2 |= {("row", p) for p in k2_row_paths(w, W)}
    k2.add(k2_dispatch(2, 1, 19, 9, 13, 50, 68, True, w_aligned=False))     # test_k2_dispatch_runs_the_mirrored_kernel
    want_k2 = {("cta", ct) for ct in (2, 8, 19, 32)} | {("v2", c, lm) for c in (2, 19) for lm in (0, 1, 2)} | \
              {("row", "staged"), ("row", "global")}
    assert k2 == want_k2, want_k2 ^ k2
    # a shape the warp-tile kernel rejects for its 9-column span, at a class count it takes
    assert not _v2_eligible(1, 19, 9, 9, 40, 32) and _v2_eligible(1, 19, 8, 8, 40, 32)
    k5 = {k5_dispatch(C, slot) for (_, C, _, _, _, _, slot, *_r) in K5_CASES}
    assert k5 == {(ct, s) for ct in (2, 8, 16, 19, 24, 32) for s in (0, 1)}
    assert {c[7] for c in K5_CASES} == {0.9, 1.0, 0.05} and {c[8] for c in K5_CASES} == {1.8, 1.0}
    k3 = set()
    for (N, K, H, W, layout, weighted, soft, off) in K3_CASES:
        for stats in (True, False):
            k3 |= set(k3_dispatch(K, layout == "vec", stats))
    assert k3 == {"fwd_v4", "bwd_stats_v4"} | {f"{d}<{kt}>" for d in ("fwd", "bwd") for kt in (4, 38, 64)}, k3
    assert {c[5] for c in K3_CASES} == {True, False} and {c[6] for c in K3_CASES} == {"dense", "zero_rows", "zero_w"}


# ==================================================================================================================== GPU
@pytest.fixture(scope="module")
def lib():
    from rnd_semantic_segmentation_b200 import _lib
    _lib.load()
    return _lib


def _bits(t):
    return t.detach().contiguous().view(torch.int32 if t.element_size() == 4 else torch.int16)


def _k2_run(lib, variant, x, lab, ign, T, go):
    """forward (with gradient), fp32 backward and packed backward on one workspace."""
    lib.upsample_ce_set_variant(variant)
    try:
        N, C, h, w = x.shape
        size = tuple(lab.shape[-2:])
        out2, ws = lib.upsample_ce_forward(x, lab, ign, 1.0 / T, True)
        g32 = lib.upsample_ce_backward(ws, out2, (N, C, h, w), size, 1.0 / T, go)
        gOt, bias = lib.upsample_ce_backward_packed(ws, out2, (N, C, h, w), size, 1.0 / T, go, True)
        torch.cuda.synchronize()
        planes = gOt.view(-1)[:N * C * h * w].view(N, C, h, w)
        return out2.cpu(), g32, planes, bias
    finally:
        lib.upsample_ce_set_variant(1)


def _check_k2(name, out2, g32, planes, bias, ref, go, warp_tile):
    loss, grad, n_valid, S, A, U, U2 = ref
    U = U2 if warp_tile else U
    assert int(out2[1].item()) == n_valid and out2[1].item() == float(n_valid), (out2[1].item(), n_valid)
    if n_valid:
        r = _record(f"{name}.loss", torch.tensor(abs(out2[0].item() - loss.item())), torch.tensor(EPS * S.item()))
        assert r <= K2_LOSS_K, f"loss {out2[0].item()!r} vs {loss.item()!r}: {r:.3g} x 2^-24 S"
    else:
        assert math.isnan(out2[0].item())
    r = _record(f"{name}.grad", ((g32.cpu().double() - go * grad).abs() - go * U).clamp_min(0), EPS * go * A)
    assert r <= K2_GRAD_K, f"gradient: {r:.3g} x 2^-24 A"
    # the packed planes are bf16(round to nearest even) of the same fp32 values; the bias is their class sums
    assert torch.equal(_bits(planes), _bits(g32.to(torch.bfloat16)))
    gsum = g32.cpu().double().sum((0, 2, 3))
    r = _record(f"{name}.bias", (bias.cpu().double() - gsum).abs(), EPS * g32.cpu().double().abs().sum((0, 2, 3)))
    assert r <= K2_BIAS_K, f"bias: {r:.3g} x 2^-24 sum|g|"


@gpu
@pytest.mark.parametrize("case", K2_CASES, ids=_case_id)
def test_k2_against_fp64(lib, case):
    x, lab, ign, T = k2_inputs(case, seed=sum(case[1:6]))
    ref = k2_reference(x, lab, ign, T)
    xc, lc = x.cuda(), lab.cuda()
    go = torch.tensor([0.75], device="cuda")
    N, C, h, w, H, W, ldt = case[:7]
    for variant in (0, 2):
        out2, g32, planes, bias = _k2_run(lib, variant, xc, lc, ign, T, go)
        warp_tile = k2_dispatch(variant, N, C, h, w, H, W, ldt == U8)[0] == "v2"
        _check_k2(f"k2.v{variant}", out2, g32, planes, bias, ref, 0.75, warp_tile)
        again = _k2_run(lib, variant, xc, lc, ign, T, go)                    # run to run bit-identical
        assert torch.equal(_bits(again[0]), _bits(out2)) and torch.equal(_bits(again[1]), _bits(g32))
        assert torch.equal(_bits(again[2]), _bits(planes)) and torch.equal(_bits(again[3]), _bits(bias))
        lib.upsample_ce_set_variant(variant)
        try:                                                                 # forward-only instantiation: the same loss
            out2_ng, _ = lib.upsample_ce_forward(xc, lc, ign, 1.0 / T, False)
        finally:
            lib.upsample_ce_set_variant(1)
        assert torch.equal(_bits(out2_ng.cpu()), _bits(out2))


@gpu
@pytest.mark.parametrize("ldt", [torch.int64, torch.uint8])
@pytest.mark.parametrize("C", [2, 8, 19])
def test_k2_all_ignored_gives_zero_gradient(lib, ldt, C):
    """No valid label: loss NaN (as PyTorch), and every gradient output +0 -- fp32, packed bf16 planes and bias."""
    x = torch.randn(2, C, 9, 13, device="cuda")
    lab = torch.full((2, 50, 70), 255, dtype=ldt, device="cuda")
    for variant in (0, 2):
        out2, g32, planes, bias = _k2_run(lib, variant, x, lab, 255, 1.0, torch.tensor([1.0], device="cuda"))
        assert math.isnan(out2[0].item()) and out2[1].item() == 0.0
        assert (_bits(g32) == 0).all() and (_bits(planes) == 0).all() and (_bits(bias) == 0).all()


@gpu
@pytest.mark.parametrize("ldt", [torch.int64, torch.uint8])
def test_head_forward_loss_all_ignored_leaves_zero_gradients(lib, ldt):
    """A crop without a valid label must not poison the head: dX, dW and db are all zero (the loss is NaN, as PyTorch's)."""
    import rnd_semantic_segmentation_b200 as b200
    torch.manual_seed(5)
    head = b200.ASPP_Classifier_V2(128, [6, 12, 18, 24], [6, 12, 18, 24], 19).cuda()
    x = torch.relu(torch.randn(2, 128, 17, 23, device="cuda")).requires_grad_(True)
    lab = torch.full((2, 96, 128), 255, dtype=ldt, device="cuda")
    loss, _ = head.forward_loss(x, lab)
    loss.backward()
    assert torch.isnan(loss)
    assert (_bits(x.grad) == 0).all()
    for name, p in head.named_parameters():
        assert p.grad is not None and (p.grad == 0).all() and not p.grad.isnan().any(), name


@gpu
@pytest.mark.parametrize("variant,C", [(0, 19), (2, 19), (0, 8), (2, 2)])
def test_k2_nan_logit_stays_local(lib, variant, C):
    """One NaN low-res logit: the loss is NaN (as the reference's), and the gradient of every low-res pixel that shares no output
    pixel with it stays finite and within the bar.  The warp-tile kernel carries its softmax shift from one row segment of a
    column to the next, so there a NaN may reach further down its frame: checked are the other frames."""
    N, h, w, H, W = 2, 9, 13, 50, 70
    x, lab, ign, T = k2_inputs((N, C, h, w, H, W, I64, 255, "plain", "n2", 1.0), seed=77)
    lab[lab == 255] = 0                                    # every output pixel counts
    n0, c0, i, j = 1, C // 2, 4, 6
    x0 = x.clone()
    x[n0, c0, i, j] = float("nan")
    out2, g32, _, _ = _k2_run(lib, variant, x.cuda(), lab.cuda(), ign, T, torch.tensor([1.0], device="cuda"))
    assert math.isnan(out2[0].item())
    _, grad, _, _, A, U, U2 = k2_reference(x0, lab, ign, T)  # outside the reach the NaN pixel changes nothing
    My, Mx = incidence(h, H).double(), incidence(w, W).double()
    reach_y = (My.T @ My)[i] > 0                           # source rows sharing an output row with row i
    reach_x = (Mx.T @ Mx)[j] > 0
    reach = torch.zeros(N, C, h, w, dtype=torch.bool)
    if k2_dispatch(variant, N, C, h, w, H, W, False)[0] == "v2":
        reach[n0] = True
        U = U2
    else:
        reach[n0] = (reach_y[:, None] & reach_x[None, :])
    g = g32.cpu().double()
    assert torch.isfinite(g[~reach]).all()
    r = _record(f"k2.v{variant}.grad", ((g - grad).abs() - U)[~reach].clamp_min(0), EPS * A[~reach])
    assert r <= K2_GRAD_K


@gpu
@pytest.mark.parametrize("shape", [(1, 19, 20, 24, 10, 12), (1, 2, 12, 40, 6, 20), (1, 19, 64, 64, 16, 16), (1, 8, 300, 8, 5, 8)])
def test_k2_downsampling_is_correct_or_refused(lib, shape):
    """Down-sampling (h > H or w > W) is not the workload, but must never fault or give a wrong number: either the result meets
    the bar, or the call fails cleanly with B200SegError before anything is written."""
    N, C, h, w, H, W = shape
    x, lab, ign, T = k2_inputs((N, C, h, w, H, W, I64, 255, "plain", "n2", 1.0), seed=5)
    xc, lc = x.cuda(), lab.cuda()
    L = lib.load()
    nbytes = L.b200seg_upsample_ce_workspace_bytes(N, C, h, w, H, W)
    ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    out2 = torch.full((2,), -7.0, device="cuda")
    rc = L.b200seg_upsample_ce_forward_ex(xc.data_ptr(), N, C, h, w, lc.data_ptr(), 8, H, W, ign, 1.0, 1, ws.data_ptr(), nbytes,
                                          out2.data_ptr(), lib._stream())
    torch.cuda.synchronize()
    if rc != 0:
        assert "shared memory" in L.b200seg_last_error().decode()
        assert (out2.cpu() == -7.0).all() and (ws == 0).all()
        with pytest.raises(lib.B200SegError, match="shared memory"):
            lib.upsample_ce_forward(xc, lc, ign, 1.0, True)
        return
    ref = k2_reference(x, lab, ign, T)
    go = torch.tensor([1.0], device="cuda")
    g32 = lib.upsample_ce_backward(ws, out2, (N, C, h, w), (H, W), 1.0, go)
    gOt, bias = lib.upsample_ce_backward_packed(ws, out2, (N, C, h, w), (H, W), 1.0, go, True)
    _check_k2("k2.down", out2.cpu(), g32, gOt.view(-1)[:N * C * h * w].view(N, C, h, w), bias, ref, 1.0, False)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


def _first(names, pattern):
    for n in names:
        m = re.search(pattern, n)
        if m:
            return m.groups()
    raise AssertionError(f"no kernel matching {pattern!r} in {sorted(set(names))}")


@gpu
def test_k2_dispatch_runs_the_mirrored_kernel(lib):
    """The mirror k2_dispatch names the kernel instantiation k2_forward really launches (kernel names from the profiler)."""
    cases = [(v, c) for c in K2_CASES for v in (0, 2)]
    cases.append((2, (1, 19, 9, 13, 50, 68, U8, 255, "plain", "n2", 1.0)))   # uint8 rows at an unaligned address
    seen, wants = set(), set()
    for variant, case in cases:
        N, C, h, w, H, W, ldt = case[:7]
        x, lab, ign, T = k2_inputs(case, seed=1)
        xc = x.cuda()
        lc = lab.cuda()
        unaligned = case is cases[-1][1]
        if unaligned:
            buf = torch.empty(lc.numel() + 1, dtype=torch.uint8, device="cuda")
            buf[1:] = lc.view(-1)
            lc = buf[1:].view(lab.shape)
        want = k2_dispatch(variant, N, C, h, w, H, W, ldt == U8, w_aligned=not unaligned)
        if (want, unaligned) in seen:
            continue
        seen.add((want, unaligned))
        wants.add(want)
        lib.upsample_ce_set_variant(variant)
        try:
            names = _kernel_names(lambda: lib.upsample_ce_forward(xc, lc, ign, 1.0 / T, True))
        finally:
            lib.upsample_ce_set_variant(1)
        if want[0] == "v2":
            ct, lm = _first(names, r"k2v2_upsample_ce_main<(\d+), *(?:true|false|\(bool\)\d), *(\d)>")
            assert (int(ct), int(lm)) == want[1:], (case, names)
        else:
            assert not any("k2v2_upsample_ce_main" in n for n in names), (case, names)
            ct, = _first(names, r"k2_upsample_ce_main<(\d+),")
            assert int(ct) == want[1], (case, names)
    assert len(wants) == 4 + 6


@gpu
def test_k5_and_k3_dispatch_run_the_mirrored_kernels(lib):
    seen = set()
    for (N, C, h, w, H, W, slot, clamp, T) in K5_CASES:
        want = k5_dispatch(C, slot)
        if want in seen:
            continue
        seen.add(want)
        d = torch.randn(N, 2 * C, h, w, device="cuda")
        seg = torch.randn(N, C, h, w, device="cuda")
        names = _kernel_names(lambda: lib.fada_softce_forward(d, seg, (H, W), slot, 1.0 / T, clamp, True))
        ct, sl = _first(names, r"k5_fada_softce_main<(\d+), *[^,]+, *[^,]+, *(\d)>")
        assert (int(ct), int(sl)) == want, names
    assert len(seen) == 12
    for (N, K, H, W, layout, weighted, srec, off) in K3_CASES:
        pred, soft, wts = k3_inputs((N, K, H, W, layout, weighted, srec, off), seed=3)
        for stats in (True, False):
            fwd, bwd = k3_dispatch(K, layout == "vec", stats)

            def run():
                st = _k3_forward(lib, pred, soft, wts, stats)[1]
                lib.soft_ce_backward(pred, soft, wts, torch.ones((), device="cuda"), st)
            names = _kernel_names(run)
            for want in (fwd, bwd):
                pat = {"fwd_v4": r"k3_softce_fwd_v4", "bwd_stats_v4": r"k3_softce_bwd_stats_v4"}.get(
                    want, r"k3_softce_" + want.replace("<", "<(?:").replace(">", ")>"))
                assert any(re.search(pat, n) for n in names), (want, sorted(set(names)))


# ============================================================================================================ K5
@gpu
@pytest.mark.parametrize("case", K5_CASES, ids=_case_id)
def test_k5_against_fp64(lib, case):
    N, C, h, w, H, W, slot, clamp, T = case
    g = torch.Generator().manual_seed(31 + C + h + slot)
    d = (1.5 * torch.randn(N, 2 * C, h, w, generator=g)).float()
    seg = (4.0 * torch.randn(N, C, h, w, generator=g)).float()
    loss, grad, S, A = k5_reference(d, seg, (H, W), slot, T, clamp)
    go = torch.tensor([0.5], device="cuda")
    runs = []
    for _ in range(2):
        out2, ws = lib.fada_softce_forward(d.cuda(), seg.cuda(), (H, W), slot, 1.0 / T, clamp, True)
        gd = lib.fada_softce_backward(ws, out2, (N, 2 * C, h, w), (H, W), go)
        runs.append((out2.cpu(), gd.cpu()))
    out2, gd = runs[0]
    assert torch.equal(_bits(runs[1][0]), _bits(out2)) and torch.equal(_bits(runs[1][1]), _bits(gd))
    assert out2[1].item() == N * H * W
    r = _record("k5.loss", torch.tensor(abs(out2[0].item() - loss.item())), torch.tensor(EPS * S.item()))
    assert r <= K5_LOSS_K, f"loss {out2[0].item()!r} vs {loss.item()!r}: {r:.3g} x 2^-24 S"
    r = _record("k5.grad", (gd.double() - 0.5 * grad).abs(), EPS * 0.5 * A)
    assert r <= K5_GRAD_K, f"gradient: {r:.3g} x 2^-24 A"
    out2_ng, _ = lib.fada_softce_forward(d.cuda(), seg.cuda(), (H, W), slot, 1.0 / T, clamp, False)
    assert torch.equal(_bits(out2_ng.cpu()), _bits(out2))


# ============================================================================================================ K3
def k3_inputs(case, seed):
    N, K, H, W, layout, weighted, srec, off = case
    g = torch.Generator().manual_seed(seed)
    pred = 3.0 * torch.randn(N, K, H, W, generator=g) + off
    soft = torch.softmax(2.0 * torch.randn(N, K, H, W, generator=g), 1)
    soft[:, K // 2 + 1:] = 0                       # the discriminator's empty slot
    wts = torch.rand(N, H, W, generator=g) if weighted or srec == "zero_w" else None
    if srec == "zero_rows":
        soft[:, :, ::3] = 0
    if srec == "zero_w":
        wts[:, ::2] = 0
    out = []
    for t in (pred, soft, wts):
        if t is None:
            out.append(None)
        elif layout == "off4":                     # contiguous view 4 bytes into its buffer: the scalar path
            buf = torch.empty(t.numel() + 1, device="cuda")
            buf[1:] = t.reshape(-1).cuda()
            out.append(buf[1:].view(t.shape))
        else:
            out.append(t.cuda())
    return out


def _k3_forward(lib, pred, soft, wts, want_stats):
    """(loss, per-pixel statistics or None)"""
    if want_stats:
        return lib.soft_ce_forward(pred, soft, wts, want_stats=True)
    return lib.soft_ce_forward(pred, soft, wts), None


@gpu
@pytest.mark.parametrize("case", K3_CASES, ids=_case_id)
def test_k3_against_fp64(lib, case):
    pred, soft, wts = k3_inputs(case, seed=11 + case[1] + case[2])
    loss, grad, S, A = soft_ce_reference(pred, soft, wts)
    go = torch.tensor(0.25, device="cuda")
    for stats_wanted in (True, False):
        got, stats = _k3_forward(lib, pred, soft, wts, stats_wanted)
        assert (stats is not None) == (stats_wanted and case[4] == "vec")
        g = lib.soft_ce_backward(pred, soft, wts, go, stats)
        r = _record("k3.loss", torch.tensor(abs(got.item() - loss.item())), torch.tensor(EPS * S.item()))
        assert r <= K3_LOSS_K, f"loss {got.item()!r} vs {loss.item()!r}: {r:.3g} x 2^-24 S"
        r = _record("k3.grad", (g.cpu().double() - 0.25 * grad).abs(), EPS * 0.25 * A)
        assert r <= K3_GRAD_K, f"gradient ({'stats' if stats is not None else 'recompute'}): {r:.3g} x 2^-24 A"
        again = lib.soft_ce_backward(pred, soft, wts, go, stats)
        assert torch.equal(_bits(again), _bits(g))
