"""The seam-format tail with conv3 fused in: fuse_backbone_tail(conv3=True) / install(seam=True, seam_conv3=True) run the last
Bottleneck's 1x1 conv3 as a tcgen05 GEMM whose epilogue applies the folded bn3, the residual and the relu (ops.seam_conv3_tail).

Numerics contract under test: out2 and W3 are rounded to bf16 once, the products are summed in fp32, the tail is applied to the
fp32 accumulator in the fold's order and the result is rounded once to bf16.  The forward oracle repeats exactly those roundings
with torch's fp32 convolution (TF32 off); the two sums differ only in their fp32 summation order, so a feature may land one bf16 ulp
away -- or, where the tail cancels to near zero, as far as that order difference (bounded here by 2^-20 of the summed magnitudes).
The backward oracle is fp64 with the same bf16 operands."""
import copy
import inspect
import sys
import types

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import rel_err
from test_seam_tail import FrozenBatchNorm2d, _block_and_head, _l2, make_block

import rnd_semantic_segmentation_b200 as b200
from rnd_semantic_segmentation_b200 import _lib, ops, seam


def _conv3_variant(kind, seed=41):
    """A small FrozenBatchNorm2d block whose conv3 is made ineligible for the fused GEMM in one way (or left eligible)."""
    planes = 12 if kind == "cin" else 16
    blk = make_block(64, planes, seed)
    c3 = blk.conv3
    if kind == "bias":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=True)
    elif kind == "3x3":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 3, padding=1, bias=False)
    elif kind == "groups":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 1, groups=2, bias=False)
    elif kind == "stride":
        blk.conv3 = nn.Conv2d(planes, planes * 4, 1, stride=2, bias=False)
        blk.downsample[0] = nn.Conv2d(64, planes * 4, 1, stride=2, bias=False)
    if blk.conv3 is not c3:
        torch.manual_seed(seed + 7)
        with torch.no_grad():
            blk.conv3.weight.mul_(2.0)
    return blk


# ------------------------------------------------------------------ CPU: flag, persistence, eligibility, install()
def test_conv3_flag_survives_save_load_and_deepcopy_and_follows_repeated_calls(tmp_path):
    fe = nn.Sequential(make_block(64, 16, 3))
    b200.fuse_backbone_tail(fe, conv3=True)
    state = fe[0].__dict__["forward"]
    assert state.conv3 and not state.train_bn
    path = tmp_path / "fe.pt"
    torch.save(fe, path)
    loaded = torch.load(path, weights_only=False)
    assert seam.is_fused(loaded) and loaded[0].__dict__["forward"].conv3
    clone = copy.deepcopy(fe)
    assert clone[0].__dict__["forward"].conv3 and clone[0].__dict__["forward"].block is clone[0]
    b200.fuse_backbone_tail(fe)                                   # a repeated call sets the flag to the new value
    assert not fe[0].__dict__["forward"].conv3
    b200.fuse_backbone_tail(fe, train_bn=True, conv3=True)
    assert fe[0].__dict__["forward"].conv3 and fe[0].__dict__["forward"].train_bn
    plain = nn.Sequential(make_block(64, 16, 3))
    b200.fuse_backbone_tail(plain)
    assert not plain[0].__dict__["forward"].conv3
    old = seam._FusedForward.__new__(seam._FusedForward)         # a hook pickled before the flag existed
    old.__dict__.update({k: v for k, v in state.__dict__.items() if k != "conv3"})
    assert old.conv3 is False


def test_conv3_eligibility_table():
    x = torch.zeros(1)
    assert seam._conv3_fusable(_conv3_variant("ok").conv3, x)
    for kind in ("bias", "3x3", "groups", "stride", "cin"):
        assert not seam._conv3_fusable(_conv3_variant(kind).conv3, x), kind
    conv = nn.Conv2d(16, 64, 1, bias=False)
    assert seam._conv3_fusable(conv, x)
    assert not seam._conv3_fusable(conv.half(), x)
    assert not seam._conv3_fusable(nn.Conv2d(16, 60, 1, bias=False), x)            # Cout % 8 != 0
    assert not seam._conv3_fusable(nn.Conv2d(16, 64, 1, padding=1, bias=False), x)

    class SubConv(nn.Conv2d):
        pass
    assert not seam._conv3_fusable(SubConv(16, 64, 1, bias=False), x)


@pytest.mark.parametrize("kind", ["ok", "bias", "3x3", "groups", "stride", "cin"])
def test_cpu_block_with_conv3_flag_is_stock(kind):
    blk = _conv3_variant(kind)
    ref = copy.deepcopy(blk)
    b200.fuse_backbone_tail(nn.Sequential(blk), conv3=True)
    x = torch.randn(2, 64, 9, 13)
    assert torch.equal(blk(x), ref(x))


def test_install_seam_conv3_wraps_the_factory_with_the_flag(monkeypatch):
    core = types.ModuleType("core"); models = types.ModuleType("core.models"); bld = types.ModuleType("core.models.build")

    def build_feature_extractor(cfg):
        return nn.Sequential(make_block(64, 16, 5))

    bld.build_feature_extractor = models.build_feature_extractor = build_feature_extractor
    bld.build_classifier = models.build_classifier = lambda cfg: "ref"
    for m in (core, models, bld):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    b200.install(seam=True)
    fn = bld.build_feature_extractor
    assert not fn(None)[0].__dict__["forward"].conv3
    b200.install(seam=True, seam_conv3=True)
    assert bld.build_feature_extractor is fn and models.build_feature_extractor is fn
    assert inspect.signature(fn) == inspect.signature(build_feature_extractor)
    st = fn(None)[0].__dict__["forward"]
    assert st.conv3 and not st.train_bn
    b200.install(seam=True, seam_train_bn=True, seam_conv3=True)
    st = fn(None)[0].__dict__["forward"]
    assert st.conv3 and st.train_bn
    b200.install(seam=True)
    assert not fn(None)[0].__dict__["forward"].conv3


# ------------------------------------------------------------------ GPU: forward against the same-rounding oracle
def _bf16_ulp(*vs):
    """bf16 ulp at the larger of |v| over the given tensors: the spacing above it (2^-133 for zero / subnormals)."""
    a = torch.stack([v.detach().float().abs() for v in vs]).amax(0)
    e = torch.floor(torch.log2(a.clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def _op_inputs(N, Cin, Cout, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    out2 = torch.relu(torch.randn(N, Cin, h, w, generator=g)).cuda()
    identity = torch.randn(N, Cout, h, w, generator=g).cuda()
    W = (torch.randn(Cout, Cin, 1, 1, generator=g) * (2.0 / Cin) ** 0.5).cuda()
    scale = (0.5 + torch.rand(Cout, generator=g)).cuda()
    bias = (0.1 * torch.randn(Cout, generator=g)).cuda()
    return out2, identity, W, scale, bias


def _no_tf32():
    class _Ctx:
        def __enter__(self):
            self.saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
            torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False

        def __exit__(self, *a):
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved
    return _Ctx()


def _oracle(out2, identity, W, scale, bias):
    """(y fp32 before the bf16 cast, magnitude of the summed terms) with the fused path's roundings."""
    s, b = scale.view(1, -1, 1, 1), bias.view(1, -1, 1, 1)
    with _no_tf32(), torch.no_grad():
        xb, wb = out2.to(torch.bfloat16).float(), W.to(torch.bfloat16).float()
        acc = F.conv2d(xb, wb)
        mag = F.conv2d(xb.abs(), wb.abs()) * s.abs() + b.abs() + identity.abs()
    return torch.relu((acc * s + b) + identity), mag


def _check_against_oracle(y, out2, identity, W, scale, bias):
    ref, mag = _oracle(out2, identity, W, scale, bias)
    refb = ref.to(torch.bfloat16)
    diff = (y.float() - refb.float()).abs()
    ulp = _bf16_ulp(refb, y)
    assert (diff <= ulp + mag * 2.0 ** -20).all(), float((diff / (ulp + mag * 2.0 ** -20)).max())
    frac = (diff > 0).float().mean().item()
    print(f"vs same-rounding oracle: max {float((diff / ulp).max()):.2f} ulp, {frac:.2e} of the features differ")
    assert frac <= 1e-3
    return frac


SHAPES = [(8, 512, 2048, 64, 128), (2, 512, 2048, 65, 129), (3, 512, 2048, 7, 9), (1, 512, 2048, 33, 65), (2, 64, 256, 33, 47)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_forward_against_same_rounding_oracle_and_stock(shape):
    N, Cin, Cout, h, w = shape
    out2, identity, W, scale, bias = _op_inputs(N, Cin, Cout, h, w, 7)
    y = b200.seam_conv3_tail(out2, identity, W, scale, bias)
    assert y.dtype == torch.bfloat16 and y.shape == (N, Cout, h, w) and y.is_contiguous(memory_format=torch.channels_last)
    _check_against_oracle(y, out2, identity, W, scale, bias)
    for tf32 in (False, True):                                   # the stock block: fp32 conv3 (cuDNN, TF32 on or off)
        saved = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = tf32
        try:
            stock = torch.relu(F.conv2d(out2, W) * scale.view(1, -1, 1, 1) + bias.view(1, -1, 1, 1) + identity)
        finally:
            torch.backends.cudnn.allow_tf32 = saved
        sb = stock.to(torch.bfloat16)
        d = (y.float() - sb.float()).abs()
        l2 = _l2(y.float(), stock)
        print(f"vs stock (tf32={tf32}): max {float((d / _bf16_ulp(sb, y)).max()):.1f} ulp, "
              f"{(d > 0).float().mean().item():.3e} differ, rel L2 {l2:.2e}")
        assert l2 <= 2.0 ** -8


@pytest.mark.gpu
@pytest.mark.parametrize("downsample", [True, False])
def test_small_block_forward(downsample):
    blk = make_block(64 if downsample else 256, 64, 51, downsample=downsample).cuda()
    g = torch.Generator().manual_seed(52)
    x = torch.relu(torch.randn(2, blk.conv1.in_channels, 21, 30, generator=g)).cuda()
    with torch.no_grad():
        out2 = blk.relu(blk.bn2(blk.conv2(blk.relu(blk.bn1(blk.conv1(x))))))
        identity = blk.downsample(x) if downsample else x
        stock = blk(x)
    scale, bias = seam._fold(blk.bn3, "frozen")
    b200.fuse_backbone_tail(nn.Sequential(blk), conv3=True)
    with torch.no_grad():
        y = blk(x)
    _check_against_oracle(y, out2, identity, blk.conv3.weight, scale, bias)
    assert _l2(y.float(), stock) <= 2.0 ** -8


# ------------------------------------------------------------------ GPU: backward against fp64 with the same roundings
def _grad_oracle(dy, y, out2, W, scale):
    g = (dy.double() * (y > 0).double())
    wp = (scale.view(-1, 1, 1, 1) * W).to(torch.bfloat16).double()                  # bf16(scale * W3), as the data gradient
    d_out2 = torch.einsum("nohw,oi->nihw", g, wp[:, :, 0, 0])
    dW = scale.double().view(-1, 1) * torch.einsum("nohw,nihw->oi", g, out2.to(torch.bfloat16).double())
    return d_out2, dW.view_as(W), g


def _ratio(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [SHAPES[0], SHAPES[1], SHAPES[2], SHAPES[4]], ids=lambda s: "x".join(map(str, s)))
def test_backward_against_fp64_oracle(shape):
    N, Cin, Cout, h, w = shape
    out2, identity, W, scale, bias = _op_inputs(N, Cin, Cout, h, w, 9)
    out2.requires_grad_(True); identity.requires_grad_(True); W.requires_grad_(True)
    y = b200.seam_conv3_tail(out2, identity, W, scale, bias)
    dy = (torch.randn(y.shape, generator=torch.Generator().manual_seed(10)).cuda()
          .to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
    y.backward(dy)
    d_out2, dW, g = _grad_oracle(dy, y.detach(), out2.detach(), W.detach(), scale)
    errs = {"out2": _ratio(out2.grad, d_out2), "weight": _ratio(W.grad, dW)}
    print("backward vs fp64:", errs)
    assert max(errs.values()) <= 1e-3
    assert torch.equal(identity.grad, g.float())                 # didentity = g exactly


@pytest.mark.gpu
def test_backward_need_flags_and_no_grad_saves_nothing():
    out2, identity, W, scale, bias = _op_inputs(2, 64, 256, 17, 23, 11)
    dy = torch.randn(2, 256, 17, 23, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    full = [t.clone().requires_grad_(True) for t in (out2, identity, W)]
    b200.seam_conv3_tail(*full, scale, bias).backward(dy)
    for need in ((False, True, True), (True, True, False), (False, False, True), (True, False, False), (False, True, False)):
        ts = [t.clone().requires_grad_(n) for t, n in zip((out2, identity, W), need)]
        b200.seam_conv3_tail(*ts, scale, bias).backward(dy)
        for t, f, n in zip(ts, full, need):
            assert (t.grad is None) == (not n)
            if n:
                assert torch.equal(t.grad, f.grad)
    saved = []
    with torch.autograd.graph.saved_tensors_hooks(lambda t: saved.append(t) or t, lambda t: t):
        with torch.no_grad():
            y0 = b200.seam_conv3_tail(*full, scale, bias)
        assert not saved and y0.grad_fn is None
        y1 = b200.seam_conv3_tail(*full, scale, bias)
    assert torch.equal(y0, y1)
    c_bytes = 2 * 256 * 17 * 23 * 4                              # conv3's fp32 output is never kept
    assert saved and all(t.numel() * t.element_size() != c_bytes for t in saved)


# ------------------------------------------------------------------ GPU: determinism and CUDA graphs
@pytest.mark.gpu
def test_run_to_run_bit_identical_and_graph_replay():
    out2, identity, W, scale, bias = _op_inputs(2, 512, 2048, 33, 47, 13)
    dy = torch.randn(2, 2048, 33, 47, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)

    def step():
        y, ws = _lib.seam_conv3_forward(out2, identity, W, scale, bias)
        return (y,) + _lib.seam_conv3_backward(dy, y, ws, scale, 512)

    a, b = step(), step()
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for t in static:
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for u, v in zip(static, a):
        assert torch.equal(u, v)


# ------------------------------------------------------------------ GPU: ineligible blocks and end to end
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bias", "3x3", "groups", "stride", "cin", "batch"])
def test_ineligible_conv3_matches_the_flag_off(kind, monkeypatch):
    if kind == "batch":
        blk = make_block(64, 16, 61, norm=nn.BatchNorm2d).train()
    else:
        blk = _conv3_variant(kind)
    a, b = copy.deepcopy(blk).cuda(), copy.deepcopy(blk).cuda()
    train_bn = kind == "batch"
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)       # (cuDNN's weight gradients may use atomics)
    b200.fuse_backbone_tail(nn.Sequential(a), train_bn=train_bn)
    b200.fuse_backbone_tail(nn.Sequential(b), train_bn=train_bn, conv3=True)
    monkeypatch.setattr(ops, "seam_conv3_tail", lambda *args: pytest.fail("ineligible conv3 took the fused GEMM"))
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


def _train_step(block, head, x, labels):
    for p in list(block.parameters()) + list(head.parameters()):
        p.grad = None
    xg = x.clone().requires_grad_(True)
    feat = block(xg)
    loss, _ = head.forward_loss(feat, labels)
    loss.backward()
    return dict(loss=loss.detach(), feat=feat.detach(), x=xg.grad,
                convs={n: p.grad.clone() for n, p in block.named_parameters() if p.requires_grad},
                head=[p.grad.clone() for p in head.parameters()])


@pytest.mark.gpu
def test_block_plus_head_train_step_against_stock(monkeypatch):
    blk, head, x, labels = _block_and_head(FrozenBatchNorm2d)
    stock = _train_step(blk, head, x, labels)
    calls = []
    real = ops.seam_conv3_tail
    monkeypatch.setattr(ops, "seam_conv3_tail", lambda *a: calls.append(1) or real(*a))
    fe = nn.Sequential(blk)
    b200.fuse_backbone_tail(fe, conv3=True)
    fused = _train_step(blk, head, x, labels)
    assert calls and fused["feat"].dtype == torch.bfloat16 and fused["feat"].is_contiguous(memory_format=torch.channels_last)
    errs = {"loss": abs(fused["loss"].item() - stock["loss"].item()) / abs(stock["loss"].item()),
            "head": max(rel_err(a, b) for a, b in zip(fused["head"], stock["head"])),
            "x": _l2(fused["x"], stock["x"]),
            **{"l2 " + n: _l2(fused["convs"][n], g) for n, g in stock["convs"].items()}}
    print("fused conv3 vs stock:", errs)
    assert errs["loss"] <= 2e-4 and errs["head"] <= 1e-2
    for k in ("l2 conv1.weight", "l2 conv2.weight", "l2 conv3.weight", "l2 downsample.0.weight"):
        assert errs[k] <= 2.0 ** -7, k
    # the block input's gradient is the sum of conv1's and downsample's data gradients, which largely cancel: its relative error
    # is about ten times that of either path (2.9e-2 on a B200, against 2-3e-3 for the weight gradients)
    assert errs["x"] <= 2.0 ** -4
    with torch.no_grad():                                         # eval: the same features with and without autograd
        assert torch.equal(blk(x), fused["feat"])
    b200.unfuse_backbone_tail(fe)
