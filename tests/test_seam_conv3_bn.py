"""conv3 under batch statistics: fuse_backbone_tail(train_bn=True, conv3_batch=True) / install(seam=True, seam_train_bn=True,
seam_conv3_batch=True) run a training-mode BatchNorm2d / SyncBatchNorm block's 1x1 conv3 as a tcgen05 GEMM that writes conv3's
output c once (fp32 NCHW) and bn3's per-rank statistics from its accumulator (ops.seam_conv3_tail_bn).

Numerics contract under test: out2 and W3 are rounded to bf16 once and summed in fp32; the statistics are those of the stored c;
the batch tail is the unchanged seam_tail_bn_forward; in the backward dc is rounded once to bf16 before conv3's two GEMMs.  The
c oracle is torch's fp32 convolution of the same bf16 operands (TF32 off), whose summation order differs: each element within
2^-20 of the summed magnitudes, plus 2^-24 of them per 16-deep MMA k-step -- the tensor cores' fp32 accumulation can lose up to
an ulp of the running sum per step, which shows where one large product comes first (the 10^3-sigma channel with Cin = 512 was
measured at 1.57e-6 = 2^-19.3 of its summed magnitudes on a B200).  The backward oracle is fp64 with the same roundings."""
import copy
import datetime
import inspect
import itertools
import sys
import types

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import rel_err
from test_seam_conv3 import _bf16_ulp, _no_tf32, _ratio, _train_step
from test_seam_tail import _block_and_head, _l2, make_block

import rnd_semantic_segmentation_b200 as b200
from rnd_semantic_segmentation_b200 import _lib, ops, seam


def _bn_block(kind="ok", seed=71, momentum=0.1):
    """A small training-mode BatchNorm2d block whose conv3 is eligible for the GEMM, or made ineligible in one way."""
    planes = 12 if kind == "cin" else 16
    blk = make_block(64, planes, seed, norm=nn.BatchNorm2d).train()
    if kind == "bias":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=True)
    elif kind == "3x3":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 3, padding=1, bias=False)
    elif kind == "groups":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 1, groups=2, bias=False)
    elif kind == "stride":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 1, stride=2, bias=False)
        blk.downsample[0] = nn.Conv2d(64, planes * 4, 1, stride=2, bias=False)
    for m in blk.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.momentum = momentum
    return blk


# ------------------------------------------------------------------ CPU: flag, persistence, install()
def test_conv3_batch_flag_survives_save_load_and_deepcopy_and_follows_repeated_calls(tmp_path):
    fe = nn.Sequential(_bn_block())
    b200.fuse_backbone_tail(fe, train_bn=True, conv3_batch=True)
    state = fe[0].__dict__["forward"]
    assert state.conv3_batch and state.train_bn and not state.conv3
    path = tmp_path / "fe.pt"
    torch.save(fe, path)
    loaded = torch.load(path, weights_only=False)
    assert seam.is_fused(loaded) and loaded[0].__dict__["forward"].conv3_batch
    clone = copy.deepcopy(fe)
    assert clone[0].__dict__["forward"].conv3_batch and clone[0].__dict__["forward"].block is clone[0]
    b200.fuse_backbone_tail(fe, train_bn=True)                    # a repeated call sets the flag to its new value
    assert not fe[0].__dict__["forward"].conv3_batch
    b200.fuse_backbone_tail(fe, train_bn=True, conv3=True, conv3_batch=True)
    st = fe[0].__dict__["forward"]
    assert st.conv3_batch and st.conv3 and st.train_bn
    old = seam._FusedForward.__new__(seam._FusedForward)         # a hook pickled before the flag existed
    old.__dict__.update({k: v for k, v in state.__dict__.items() if k != "conv3_batch"})
    assert old.conv3_batch is False


def test_install_seam_conv3_batch_wraps_the_factory_with_the_flag(monkeypatch):
    core = types.ModuleType("core"); models = types.ModuleType("core.models"); bld = types.ModuleType("core.models.build")

    def build_feature_extractor(cfg):
        return nn.Sequential(_bn_block(seed=5))

    bld.build_feature_extractor = models.build_feature_extractor = build_feature_extractor
    bld.build_classifier = models.build_classifier = lambda cfg: "ref"
    for m in (core, models, bld):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    b200.install(seam=True, seam_train_bn=True)
    fn = bld.build_feature_extractor
    assert not fn(None)[0].__dict__["forward"].conv3_batch
    b200.install(seam=True, seam_train_bn=True, seam_conv3_batch=True)
    assert bld.build_feature_extractor is fn and models.build_feature_extractor is fn
    assert inspect.signature(fn) == inspect.signature(build_feature_extractor)
    st = fn(None)[0].__dict__["forward"]
    assert st.conv3_batch and st.train_bn and not st.conv3
    b200.install(seam=True)
    st = fn(None)[0].__dict__["forward"]
    assert not st.conv3_batch and not st.train_bn


@pytest.mark.parametrize("momentum", [0.1, None])
def test_cpu_block_with_conv3_batch_flag_is_stock(momentum):
    blk = _bn_block(momentum=momentum)
    ref = copy.deepcopy(blk)
    b200.fuse_backbone_tail(nn.Sequential(blk), train_bn=True, conv3_batch=True)
    x = torch.randn(2, 64, 9, 13)
    assert torch.equal(blk(x), ref(x))
    for a, b in zip(blk.buffers(), ref.buffers()):
        assert torch.equal(a, b)


# ------------------------------------------------------------------ GPU: c and its statistics
def _conv3_inputs(N, Cin, Cout, h, w, seed, nan=False, special=False):
    """out2 / W3; ``special``: channel 0 of c offset by ~10^3 sigma (input channel 0 is constant 1, W3[0, 0] = 1000) and channel
    1 of c constant (W3[1] = 0.5 e_0); ``nan``: one NaN pixel of out2."""
    g = torch.Generator().manual_seed(seed)
    out2 = torch.relu(torch.randn(N, Cin, h, w, generator=g))
    W = torch.randn(Cout, Cin, 1, 1, generator=g) * (2.0 / Cin) ** 0.5
    if special:
        out2[:, 0] = 1.0
        W[0, 0] = 1000.0
        W[1] = 0.0
        W[1, 0] = 0.5
    if nan:
        out2[0, 3, h // 2, w // 3] = float("nan")
    return out2.cuda(), W.cuda()


def _oracle_c(out2, W):
    with _no_tf32(), torch.no_grad():
        xb, wb = out2.to(torch.bfloat16).float(), W.to(torch.bfloat16).float()
        return F.conv2d(xb, wb), F.conv2d(xb.abs(), wb.abs())


def _check_record(rec, c, what):
    C = c.shape[1]
    c64 = c.double().transpose(0, 1).reshape(C, -1)
    mean64, var64 = c64.mean(1), c64.var(1, unbiased=False)
    P = c64.shape[1]
    assert torch.equal(rec[0], torch.full_like(rec[0], float(P))), what
    mean, var = rec[1], rec[2] / P
    ok = ~torch.isnan(mean64)
    assert torch.equal(torch.isnan(mean), ~ok) and torch.equal(torch.isnan(var), ~ok), what
    sd = var64.sqrt()
    dm, dv = (mean - mean64).abs()[ok], (var - var64).abs()[ok]
    assert (dm <= 1e-6 * (mean64.abs() + sd)[ok]).all(), (what, float((dm / (mean64.abs() + sd)[ok]).max()))
    assert (dv <= 1e-5 * var64[ok]).all(), (what, float((dv / var64[ok].clamp_min(1e-300)).max()))


STAT_SHAPES = [(1, 64, 256, 65, 129), (2, 40, 72, 17, 23), (3, 512, 2048, 7, 9), (2, 64, 256, 1, 1), (1, 64, 256, 8, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("nan", [False, True])
@pytest.mark.parametrize("shape", STAT_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_stored_c_and_epilogue_statistics(shape, nan):
    N, Cin, Cout, h, w = shape
    out2, W = _conv3_inputs(N, Cin, Cout, h, w, 3, nan, special=True)
    c, rec, ws = _lib.seam_conv3_bn_forward(out2, W)
    assert c.shape == (N, Cout, h, w) and c.dtype == torch.float32 and rec.shape == (3, Cout) and rec.dtype == torch.float64
    ref, mag = _oracle_c(out2, W)
    assert torch.equal(torch.isnan(c), torch.isnan(ref))
    fin = ~torch.isnan(ref)
    assert bool(nan) == bool((~fin).any())
    bar = 2.0 ** -20 + -(-Cin // 16) * 2.0 ** -24
    assert ((c - ref).abs()[fin] <= mag[fin] * bar).all(), float(((c - ref).abs() / mag.clamp_min(1e-30))[fin].max())
    _check_record(rec, c, "epilogue vs fp64")
    _check_record(_lib.bn_stats(c), c, "bn_stats vs fp64")
    if not nan:
        sd = (rec[2] / rec[0]).sqrt()
        assert float(rec[1][0] / sd[0]) > 500.0                   # the offset channel: |mean| >> sigma
        assert float(rec[2][1]) == 0.0                           # the constant channel


# ------------------------------------------------------------------ GPU: forward
def _op_args(Cout, seed, affine=True):
    g = torch.Generator().manual_seed(seed)
    weight = (0.5 + torch.rand(Cout, generator=g)).cuda() if affine else None
    bias = (0.1 * torch.randn(Cout, generator=g)).cuda() if affine else None
    return weight, bias


def _identity(N, Cout, h, w, seed):
    return torch.randn(N, Cout, h, w, generator=torch.Generator().manual_seed(seed)).cuda()


FWD_SHAPES = [(8, 512, 2048, 64, 128), (1, 64, 256, 65, 129), (2, 40, 72, 17, 23)]


@pytest.mark.gpu
@pytest.mark.parametrize("momentum", [0.1, None])
@pytest.mark.parametrize("shape", FWD_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_forward_against_tail_and_same_rounding_oracle(shape, momentum):
    N, Cin, Cout, h, w = shape
    out2, W = _conv3_inputs(N, Cin, Cout, h, w, 21)
    identity = _identity(N, Cout, h, w, 22)
    weight, bias = _op_args(Cout, 23)
    rm, rv = 0.1 * torch.randn(Cout, device="cuda"), 1.0 + torch.rand(Cout, device="cuda")
    nbt = torch.tensor(3, dtype=torch.int64, device="cuda")
    ref_bn = nn.BatchNorm2d(Cout, momentum=momentum).cuda().train()
    with torch.no_grad():
        ref_bn.running_mean.copy_(rm); ref_bn.running_var.copy_(rv); ref_bn.num_batches_tracked.copy_(nbt)
        ref_bn.weight.copy_(weight); ref_bn.bias.copy_(bias)
    y = b200.seam_conv3_tail_bn(out2, identity, W, weight, bias, rm, rv, nbt, momentum, 1e-5)
    assert y.dtype == torch.bfloat16 and y.shape == (N, Cout, h, w) and y.is_contiguous(memory_format=torch.channels_last)
    assert int(nbt) == 4
    # y is the unchanged batch tail on the stored c with the statistics the op combined
    c, rec, _ = _lib.seam_conv3_bn_forward(out2, W)
    mean, invstd, _ = _lib.bn_combine_stats(rec, 1e-5)
    assert torch.equal(y, _lib.seam_tail_bn_forward(c, identity, mean, invstd, weight, bias))
    # the same-rounding oracle: bf16 operands -> fp32 conv -> training batch_norm -> + identity -> relu -> bf16
    acc, mag_c = _oracle_c(out2, W)
    with torch.no_grad(), _no_tf32():
        want = torch.relu(ref_bn(acc) + identity)
        m, v = acc.mean((0, 2, 3)), acc.var((0, 2, 3), unbiased=False)
        k = (weight / torch.sqrt(v + 1e-5)).abs().view(1, -1, 1, 1)
        mag = mag_c * k + (m.view(1, -1, 1, 1).abs() * k) + bias.abs().view(1, -1, 1, 1) + identity.abs()
    wantb = want.to(torch.bfloat16)
    diff = (y.float() - wantb.float()).abs()
    assert (diff <= _bf16_ulp(wantb, y) + mag * 2.0 ** -20).all()
    frac = (diff > 0).float().mean().item()
    print(f"vs same-rounding oracle: {frac:.2e} of the features differ")
    assert frac <= 1e-4
    assert rel_err(rm, ref_bn.running_mean) <= 1e-6 and rel_err(rv, ref_bn.running_var) <= 1e-6
    assert torch.equal(nbt, ref_bn.num_batches_tracked)


# ------------------------------------------------------------------ GPU: backward against fp64 with the same roundings
def _bwd_case(shape, seed, affine=True):
    N, Cin, Cout, h, w = shape
    out2, W = _conv3_inputs(N, Cin, Cout, h, w, seed, special=True)
    identity = _identity(N, Cout, h, w, seed + 1)
    weight, bias = _op_args(Cout, seed + 2, affine)
    dy = (torch.randn((N, Cout, h, w), generator=torch.Generator().manual_seed(seed + 3)).cuda()
          .to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
    return out2, identity, W, weight, bias, dy


def _dc_fp64(dy, y, c, mean, invstd, weight):
    g = dy.double() * (y > 0).double()
    xmu = c.double() - mean.double().view(1, -1, 1, 1)
    M = c.numel() / c.shape[1]
    sg, sx = g.sum((0, 2, 3)).view(1, -1, 1, 1), (g * xmu).sum((0, 2, 3)).view(1, -1, 1, 1)
    iv = invstd.double().view(1, -1, 1, 1)
    gam = 1.0 if weight is None else weight.double().view(1, -1, 1, 1)
    return (g - sg / M - xmu * iv * iv * sx / M) * iv * gam, g


@pytest.mark.gpu
@pytest.mark.parametrize("affine", [True, False])
@pytest.mark.parametrize("shape", FWD_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_backward_against_fp64_oracle(shape, affine):
    out2, identity, W, weight, bias, dy = _bwd_case(shape, 31, affine)
    leaves = [out2, identity, W] + ([weight, bias] if affine else [])
    leaves = [t.clone().requires_grad_(True) for t in leaves]
    xa, ia, wa = leaves[:3]
    ga, ba = (leaves[3], leaves[4]) if affine else (None, None)
    y = b200.seam_conv3_tail_bn(xa, ia, wa, ga, ba, None, None, None, 0.1, 1e-5)
    y.backward(dy)
    c, rec, _ = _lib.seam_conv3_bn_forward(out2, W)
    mean, invstd, _ = _lib.bn_combine_stats(rec, 1e-5)
    dc, g = _dc_fp64(dy, y.detach(), c, mean, invstd, weight)
    dcb = dc.float().to(torch.bfloat16).double()
    d_out2 = torch.einsum("nohw,oi->nihw", dcb, W.to(torch.bfloat16).double()[:, :, 0, 0])
    dW = torch.einsum("nohw,nihw->oi", dcb, out2.to(torch.bfloat16).double()).view_as(W)
    errs = {"out2": _ratio(xa.grad, d_out2), "conv weight": _ratio(wa.grad, dW)}
    print("backward vs fp64:", errs)
    assert max(errs.values()) <= 2e-5
    assert torch.equal(ia.grad, g.float())
    if affine:
        _, _, gw, gb = torch.batch_norm_backward_reduce(g.float().contiguous(), c, mean, invstd, weight, True, True, True)
        assert rel_err(ga.grad, gw) <= 1e-5 and rel_err(ba.grad, gb) <= 1e-5


@pytest.mark.gpu
def test_every_subset_of_needed_gradients_and_no_grad():
    shape = (2, 64, 256, 17, 23)
    out2, identity, W, weight, bias, dy = _bwd_case(shape, 41)
    base = (out2, identity, W, weight, bias)

    def run(need, rm=None, rv=None, nbt=None):
        ts = [t.clone().requires_grad_(n) for t, n in zip(base, need)]
        y = b200.seam_conv3_tail_bn(*ts, rm, rv, nbt, 0.1, 1e-5)
        if any(need):
            y.backward(dy)
        return y, ts

    y_full, full = run((True,) * 5)
    for need in itertools.product((False, True), repeat=5):
        if not any(need) or all(need):
            continue
        y, ts = run(need)
        assert torch.equal(y, y_full)
        for t, f, n in zip(ts, full, need):
            assert (t.grad is None) == (not n)
            if n:
                assert torch.equal(t.grad, f.grad), need
    rm, rv = torch.zeros(256, device="cuda"), torch.ones(256, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    saved = []
    with torch.autograd.graph.saved_tensors_hooks(lambda t: saved.append(t) or t, lambda t: t):
        with torch.no_grad():
            y0 = b200.seam_conv3_tail_bn(*full, rm, rv, nbt, 0.1, 1e-5)
    assert not saved and y0.grad_fn is None and torch.equal(y0, y_full)
    assert int(nbt) == 1
    rm1, rv1 = torch.zeros(256, device="cuda"), torch.ones(256, device="cuda")
    _lib.bn_combine_stats(_lib.seam_conv3_bn_forward(out2, W)[1], 1e-5, 0.1, rm1, rv1)
    assert torch.equal(rm, rm1) and torch.equal(rv, rv1)                    # updated exactly once
    with pytest.raises(ValueError):
        b200.seam_conv3_tail_bn(out2[:1, :, :1, :1], identity[:1, :, :1, :1], W, weight, bias, None, None, None, 0.1, 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("shards", [[2, 2], [1, 2, 1, 1]])
def test_sharded_backward_emulates_syncbatchnorm(shards):
    """R ranks, each with its shard: the records and the backward sums gathered in rank order.  Against the unsharded batch: the
    combined statistics and sums, and the fp32 dc of the batch tail, within 1e-5; given the same gathered statistics and sums,
    the unsharded conv3 backward gives the same d_out2 and dW3 (the pixel sum over the shards) within 1e-5."""
    shape = (sum(shards), 64, 256, 33, 65)
    out2, identity, W, weight, bias, dy = _bwd_case(shape, 51)
    # the unsharded batch
    c, rec, ws = _lib.seam_conv3_bn_forward(out2, W)
    mean, invstd, count = _lib.bn_combine_stats(rec, 1e-5)
    y = _lib.seam_tail_bn_forward(c, identity, mean, invstd, weight, bias)
    sums = _lib.seam_tail_bn_backward_reduce(dy, y, c, mean, invstd)[0]
    dc = _lib.seam_tail_bn_backward(dy, y, c, mean, invstd, weight, sums, count)[0]
    # R ranks
    parts = [_lib.seam_conv3_bn_forward(t.contiguous(), W) for t in torch.split(out2, shards)]
    smean, sinv, scount = _lib.bn_combine_stats(torch.stack([p[1] for p in parts]), 1e-5)
    assert rel_err(smean, mean) <= 1e-6 and rel_err(sinv, invstd) <= 1e-6 and torch.equal(scount, count)
    ids, dys = [t.contiguous() for t in torch.split(identity, shards)], torch.split(dy, shards)
    ys = [_lib.seam_tail_bn_forward(p[0], i, smean, sinv, weight, bias) for p, i in zip(parts, ids)]
    ssums = torch.stack([_lib.seam_tail_bn_backward_reduce(d, t, p[0], smean, sinv)[0] for d, t, p in zip(dys, ys, parts)])
    assert rel_err(ssums.sum(0), sums) <= 1e-5
    sdc = torch.cat([_lib.seam_tail_bn_backward(d, t, p[0], smean, sinv, weight, ssums, scount)[0] for d, t, p in zip(dys, ys, parts)])
    assert rel_err(sdc, dc) <= 1e-5
    outs = [_lib.seam_conv3_bn_backward(d, t, p[0], smean, sinv, weight, ssums, scount, p[2], 64) for d, t, p in zip(dys, ys, parts)]
    ycat = torch.cat(ys).contiguous(memory_format=torch.channels_last)
    dx, dw, _ = _lib.seam_conv3_bn_backward(dy, ycat, c, smean, sinv, weight, ssums, scount, ws, 64)
    assert rel_err(torch.cat([o[0] for o in outs]), dx) <= 1e-5
    assert rel_err(sum(o[1] for o in outs), dw) <= 1e-5


# ------------------------------------------------------------------ GPU: block + head, ineligible blocks
def _bf16_conv3(block):
    """The stock block with conv3 computed from bf16(out2) and bf16(W3) in fp32: the forward roundings of the fused path."""
    conv = block.conv3
    conv.forward = lambda t: F.conv2d(t.to(torch.bfloat16).float(), conv.weight.to(torch.bfloat16).float())
    return block


def _errs(fused, ref):
    return {"loss": abs(fused["loss"].item() - ref["loss"].item()) / abs(ref["loss"].item()),
            "head": max(rel_err(a, b) for a, b in zip(fused["head"], ref["head"])),
            "x": _l2(fused["x"], ref["x"]),
            **{"l2 " + n: _l2(fused["convs"][n], g) for n, g in ref["convs"].items() if n.endswith("weight") and "bn" not in n}}


@pytest.mark.gpu
@pytest.mark.parametrize("momentum", [0.1, None])
def test_training_batchnorm_block_plus_head_against_stock(momentum, monkeypatch):
    """Against the stock block the loss, head gradients and block-input gradient meet the fused-conv3 bars; the conv weight
    gradients move by 3-4 % (relative L2, B200), not the fold path's 0.3 %: under batch statistics the bf16 rounding of out2 and W3
    alone moves them that far (reproduced by the stock block on the CPU with conv3 fed bf16-rounded operands), so they are held to
    2^-4 there and to 2^-7 against the stock block with exactly that forward rounding.  The running buffers likewise."""
    blk, head, x, labels = _block_and_head(norm=nn.BatchNorm2d)
    blk.train()
    for m in blk.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.momentum = momentum
    ref, same = copy.deepcopy(blk), _bf16_conv3(copy.deepcopy(blk))
    calls = []
    real = ops.seam_conv3_tail_bn
    monkeypatch.setattr(ops, "seam_conv3_tail_bn", lambda *a: calls.append(1) or real(*a))
    b200.fuse_backbone_tail(nn.Sequential(blk), train_bn=True, conv3_batch=True)
    for step in range(2):
        stock = _train_step(ref, head, x, labels)
        rounded = _train_step(same, head, x, labels)
        fused = _train_step(blk, head, x, labels)
        assert len(calls) == step + 1 and fused["feat"].dtype == torch.bfloat16
        errs, errs_same = _errs(fused, stock), _errs(fused, rounded)
        print("conv3 under batch statistics vs stock:", errs)
        print("  vs stock with bf16 conv3 operands:", errs_same)
        assert errs["loss"] <= 2e-4 and errs["head"] <= 1e-2 and errs["x"] <= 2.0 ** -4
        for k in ("l2 conv1.weight", "l2 conv2.weight", "l2 conv3.weight", "l2 downsample.0.weight"):
            assert errs[k] <= 2.0 ** -4, k
            assert errs_same[k] <= 2.0 ** -7, k
        assert errs_same["x"] <= 2.0 ** -7
    # the running buffers follow the statistics of the stored c: within 1e-5 of the stock block fed the same bf16 operands; the
    # operand rounding alone moves them from the stock fp32 block's by 1.1e-3 / 1.5e-3 (momentum 0.1 / None, max-abs over max-abs,
    # the stock block with bf16-rounded conv3 operands against the plain one on the CPU)
    for name in ("running_mean", "running_var"):
        got = getattr(blk.bn3, name)
        assert rel_err(got, getattr(same.bn3, name)) <= 1e-5, name
        assert rel_err(got, getattr(ref.bn3, name)) <= 2.0 ** -8, name
    assert torch.equal(blk.bn3.num_batches_tracked, ref.bn3.num_batches_tracked)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bias", "3x3", "groups", "stride", "cin"])
def test_ineligible_conv3_matches_train_bn_alone(kind, monkeypatch):
    blk = _bn_block(kind, 61)
    a, b = copy.deepcopy(blk).cuda(), copy.deepcopy(blk).cuda()
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)       # (cuDNN's weight gradients may use atomics)
    b200.fuse_backbone_tail(nn.Sequential(a), train_bn=True)
    b200.fuse_backbone_tail(nn.Sequential(b), train_bn=True, conv3_batch=True)
    monkeypatch.setattr(ops, "seam_conv3_tail_bn", lambda *args: pytest.fail("ineligible conv3 took the GEMM"))
    x = torch.relu(torch.randn(2, 64, 18, 27, generator=torch.Generator().manual_seed(62))).cuda()
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    ya, yb = a(xa), b(xb)
    assert ya.dtype == yb.dtype and torch.equal(ya, yb)
    dy = torch.randn(ya.shape, device="cuda").to(ya.dtype)
    ya.backward(dy)
    yb.backward(dy)
    assert torch.equal(xa.grad, xb.grad)
    for (n, p), q in zip(a.named_parameters(), b.parameters()):
        assert torch.equal(p.grad, q.grad), n
    for p, q in zip(a.buffers(), b.buffers()):
        assert torch.equal(p, q)


# ------------------------------------------------------------------ GPU: determinism and CUDA graphs
@pytest.mark.gpu
def test_run_to_run_bit_identical_and_graph_replay_matches_eager():
    shape = (2, 512, 2048, 33, 47)
    out2, identity, W, weight, bias, dy = _bwd_case(shape, 81)
    leaves = [t.clone().requires_grad_(True) for t in (out2, identity, W, weight, bias)]
    rm, rv = torch.zeros(2048, device="cuda"), torch.ones(2048, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")

    def step():
        y = b200.seam_conv3_tail_bn(*leaves, rm, rv, nbt, 0.1, 1e-5)
        return (y,) + torch.autograd.grad(y, leaves, dy)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        static = step()
    state0 = [t.clone() for t in (rm, rv, nbt)]

    def reset():
        for t, v in zip((rm, rv, nbt), state0):
            t.copy_(v)

    reset()
    graph.replay()
    torch.cuda.synchronize()
    replayed, state1 = [t.clone() for t in static], [t.clone() for t in (rm, rv, nbt)]
    reset()
    a = step()
    for u, v in zip(replayed, a):
        assert torch.equal(u, v)
    for u, v in zip(state1, (rm, rv, nbt)):
        assert torch.equal(u, v)
    reset()
    b = step()                                                    # run to run
    for u, v in zip(a, b):
        assert torch.equal(u, v)


# ------------------------------------------------------------------ two ranks: SyncBatchNorm through DDP
def _two_rank_worker(rank, world, init_file):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{init_file}", rank=rank, world_size=world,
                            timeout=datetime.timedelta(seconds=300))
    try:
        torch.manual_seed(0)
        base = nn.Sequential(make_block(256, 64, 51, norm=nn.BatchNorm2d)).train()
        stock = nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(base)).cuda()         # train_distill.py:52-53
        fused = nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(base)).cuda()
        b200.fuse_backbone_tail(fused, train_bn=True, conv3_batch=True)
        stock_ddp = DDP(stock, device_ids=[rank], find_unused_parameters=True)
        fused_ddp = DDP(fused, device_ids=[rank], find_unused_parameters=True)
        torch.manual_seed(52)
        head = b200.ASPP_Classifier_V2(256, [6, 12], [6, 12], 19).cuda()
        g = torch.Generator().manual_seed(100 + rank)                       # each rank its own shard
        x = torch.relu(torch.randn(2, 256, 17, 33, generator=g)).cuda()
        labels = torch.randint(0, 19, (2, 68, 132), generator=g).cuda()
        out = {}
        for name, model in (("stock", stock_ddp), ("fused", fused_ddp)):
            for p in list(model.parameters()) + list(head.parameters()):
                p.grad = None
            xg = x.clone().requires_grad_(True)
            feat = model(xg)
            loss, _ = head.forward_loss(feat, labels)
            loss.backward()
            bn3 = model.module[0].bn3
            out[name] = dict(loss=loss.detach(), x=xg.grad, feat=feat.detach(), head=[p.grad.clone() for p in head.parameters()],
                             params={n: p.grad.clone() for n, p in model.named_parameters()},
                             rm=bn3.running_mean.clone(), rv=bn3.running_var.clone(), gw=bn3.weight.grad.clone(),
                             gb=bn3.bias.grad.clone(), gc3=model.module[0].conv3.weight.grad.clone())
        s, f = out["stock"], out["fused"]
        assert f["feat"].dtype == torch.bfloat16
        assert abs(f["loss"].item() - s["loss"].item()) <= 2e-4 * abs(s["loss"].item())
        assert max(rel_err(a, b) for a, b in zip(f["head"], s["head"])) <= 1e-2
        assert _l2(f["x"], s["x"]) <= 2.0 ** -4
        for n, gs in s["params"].items():
            if n.endswith("conv1.weight") or n.endswith("conv2.weight") or n.endswith("conv3.weight") or "downsample.0" in n:
                assert _l2(f["params"][n], gs) <= 2.0 ** -4, n        # (see the single-rank block test)
        assert rel_err(f["rm"], s["rm"]) <= 2.0 ** -8 and rel_err(f["rv"], s["rv"]) <= 2.0 ** -8     # (see the single-rank block test)
        # identical on both ranks: the statistics (hence the running buffers) and, after DDP, the gradients
        for key in ("rm", "rv", "gw", "gb", "gc3"):
            both = [torch.empty_like(f[key]) for _ in range(world)]
            dist.all_gather(both, f[key])
            assert torch.equal(both[0], both[1]), key
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_rank_syncbatchnorm_ddp_matches_stock(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp
    mp.spawn(_two_rank_worker, args=(2, str(tmp_path / "pg_init")), nprocs=2, join=True)
