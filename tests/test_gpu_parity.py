"""-m gpu parity tests: the CUDA path (through the C ABI, via the ctypes host layer) against the oracle on the same
seeded inputs.  Bars: bit-exact for argmax labels / confusion matrices (vs the oracle's torch CUDA ops, i.e. what the
reference computes on the GPU); <= 1e-3 relative (max-abs / max-abs) for logits, losses and gradients with fp32
accumulation -- the tolerance BASELINE.json's north_star states."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import RATES, bf16_round, effective_bf16_head, make_labels, rel_err
from oracle import torch_oracle as to

pytestmark = pytest.mark.gpu
TOL = 1e-3


@pytest.fixture(scope="module")
def lib():
    from rnd_semantic_segmentation_b200 import _lib
    _lib.load()
    return _lib


# ------------------------------------------------------------------ tcgen05 GEMM core
@pytest.mark.parametrize("M,N,K,a_mn,b_mn,splits,col_hw", [
    (640, 1024, 2048, False, False, 1, 0),      # fwd shape class
    (640, 777, 2048, False, False, 1, 0),       # ragged N
    (128, 300, 64, False, False, 1, 0),         # single k-block
    (2048, 1000, 640, False, False, 1, 251),    # dgrad shape class, NCHW column map with odd hw (scalar stores)
    (2048, 1024, 640, False, False, 1, 256),    # dgrad shape class, aligned images (vector stores)
    (300, 1000, 128, False, False, 1, 200),
    (640, 2048, 5000, True, True, 3, 0),        # wgrad shape class, MN-major, split-K, ragged K
    (128, 512, 200, True, True, 1, 0),
    (100, 200, 96, False, False, 1, 0),         # ragged M
    (640, 512, 1000, True, False, 2, 0),
    (256, 512, 1000, False, True, 1, 0),
])
@pytest.mark.parametrize("share", [0, 1, 2, 3, 4])
def test_gemm_core_matches_cuda_core_reference(lib, M, N, K, a_mn, b_mn, splits, col_hw, share):
    """share: 0 = one CTA per tile; 1 / 2 = 2-CTA clusters multicasting the shared B / A tile; 3 = the same as 2 (the ABI
    value of the removed 2 x 2 clusters); 4 = CTA pairs driving one tcgen05.mma.cta_group::2 (M = 256)."""
    err, ref = lib.gemm_selftest(M, N, K, a_mn, b_mn, splits, col_hw, share)
    assert ref > 0
    assert err <= 2e-4 * ref * max(1.0, (K / 2048) ** 0.5), (err, ref)


# ------------------------------------------------------------------ materialising upsample
def test_upsample_forward_bit_exact_and_mode_report(lib):
    torch.manual_seed(0)
    x = torch.randn(2, 19, 65, 129, device="cuda")
    want = F.interpolate(x, size=(512, 1024), mode="bilinear", align_corners=True)
    matches = {m: bool(torch.equal(lib.upsample_bilinear_forward(x, (512, 1024), fma_mode=m), want)) for m in range(4)}
    print("fma modes bit-equal to ATen:", matches)
    assert matches[0], matches


@pytest.mark.parametrize("shape,size", [((2, 5, 9, 11), (50, 70)), ((1, 19, 64, 128), (512, 1024)), ((3, 2, 44, 44), (352, 352)),
                                        ((1, 3, 7, 5), (7, 5)), ((1, 4, 16, 16), (17, 31)),
                                        # streaming float4 paths (W % 4 == 0): identity, downsampling, 1-row / 1-column sources
                                        ((1, 3, 8, 8), (8, 8)), ((1, 2, 20, 24), (10, 12)), ((2, 2, 5, 6), (40, 64)),
                                        ((1, 2, 1, 7), (16, 32)), ((1, 2, 6, 1), (24, 8)), ((1, 19, 65, 129), (512, 1024))])
def test_upsample_backward_is_adjoint(lib, shape, size):
    torch.manual_seed(1)
    x = torch.randn(*shape, device="cuda", requires_grad=True)
    g = torch.randn(shape[0], shape[1], *size, device="cuda")
    want, = torch.autograd.grad(F.interpolate(x, size=size, mode="bilinear", align_corners=True), x, g)
    got = lib.upsample_bilinear_backward(g, shape[-2:])
    assert rel_err(got, want) < 1e-5
    assert torch.equal(lib.upsample_bilinear_forward(x.detach(), size), F.interpolate(x.detach(), size=size, mode="bilinear", align_corners=True))


# ------------------------------------------------------------------ K4
def _k4_case(lib, n, C, h, w, H, W, sigma, seed, p_ignore=0.1):
    g = torch.Generator().manual_seed(seed)
    logits = (sigma * torch.randn(n, C, h, w, generator=g)).cuda()
    labels = make_labels(n, H, W, C, p_ignore, seed + 1).cuda()
    want_pred = to.eval_argmax(logits, (H, W))                         # torch CUDA ops == what the reference runs
    cm, pred = lib.upsample_argmax_confusion(logits, labels, (H, W), want_pred=True, per_frame=True)
    assert torch.equal(pred, want_pred), f"{(pred != want_pred).sum().item()} of {pred.numel()} labels differ"
    for f in range(n):
        want_cm = to.confusion_matrix_bincount(C, want_pred[f].flatten(), labels[f].flatten())
        assert torch.equal(cm[f].cpu(), want_cm)
    cm_all, _ = lib.upsample_argmax_confusion(logits, labels, (H, W))
    assert torch.equal(cm_all, cm.sum(0))
    return logits, labels, pred


@pytest.mark.parametrize("n,C,h,w,H,W", [(1, 19, 64, 128, 1024, 2048), (2, 19, 65, 129, 512, 1024), (3, 2, 44, 44, 352, 352),
                                        (1, 7, 9, 11, 50, 70), (2, 19, 33, 17, 100, 131), (1, 30, 8, 8, 64, 64), (1, 19, 16, 16, 16, 16)])
@pytest.mark.parametrize("sigma", [1.0, 0.01])
def test_k4_argmax_and_confusion_bit_exact(lib, n, C, h, w, H, W, sigma):
    _k4_case(lib, n, C, h, w, H, W, sigma, seed=100 + C + h)


def test_k4_exact_ties_and_near_ties(lib):
    """Adversarial logits: identical classes (exact ties -> first index) and pairs one ulp apart."""
    torch.manual_seed(3)
    base = torch.randn(1, 1, 16, 32).repeat(1, 19, 1, 1)
    base[:, 5] = torch.nextafter(base[:, 5], torch.full_like(base[:, 5], 10.0))
    base[:, 11] = base[:, 5]
    logits = base.cuda()
    labels = make_labels(1, 128, 256, 19, 0.2, 9).cuda()
    want = to.eval_argmax(logits, (128, 256))
    cm, pred = lib.upsample_argmax_confusion(logits, labels, (128, 256), want_pred=True)
    assert torch.equal(pred, want)
    assert torch.equal(cm.cpu(), to.confusion_matrix_bincount(19, want.flatten(), labels.flatten()))


def test_k4_all_ignored_and_accumulate(lib):
    logits = torch.randn(1, 19, 8, 8, device="cuda")
    labels = torch.full((1, 64, 64), 255, dtype=torch.int64, device="cuda")
    cm, _ = lib.upsample_argmax_confusion(logits, labels, (64, 64))
    assert int(cm.sum()) == 0
    labels2 = make_labels(1, 64, 64, 19, 0.0, 4).cuda()
    cm, _ = lib.upsample_argmax_confusion(logits, labels2, (64, 64), cm=cm)
    cm, _ = lib.upsample_argmax_confusion(logits, labels2, (64, 64), cm=cm)
    assert int(cm.sum()) == 2 * 64 * 64


def test_confusion_from_pred_matches_oracle(lib):
    g = torch.Generator().manual_seed(5)
    pd = torch.randint(0, 19, (3, 77, 91), generator=g).cuda()
    gt = make_labels(3, 77, 91, 19, 0.2, 6).cuda()
    want = to.confusion_matrix_bincount(19, pd.flatten(), gt.flatten())
    assert torch.equal(lib.confusion_from_pred(pd.flatten().clone(), gt.flatten(), 19).cpu(), want)
    small = slice(0, 500)
    assert torch.equal(lib.confusion_from_pred(pd.flatten()[small].clone(), gt.flatten()[small].contiguous(), 19).cpu(),
                       to.confusion_matrix_loop(19, pd.flatten()[small].cpu(), gt.flatten()[small].cpu()))


# ------------------------------------------------------------------ K2
@pytest.mark.parametrize("n,C,h,w,H,W,T", [(2, 19, 65, 129, 512, 1024, 1.0), (1, 19, 64, 128, 512, 1024, 1.8), (3, 2, 44, 44, 352, 352, 1.0),
                                          (1, 7, 9, 11, 50, 70, 1.0), (2, 19, 33, 17, 100, 131, 1.8), (1, 19, 16, 16, 16, 16, 1.0),
                                          (1, 30, 8, 8, 64, 64, 1.0)])
def test_k2_upsample_ce_forward_backward(lib, n, C, h, w, H, W, T):
    g = torch.Generator().manual_seed(7 + C + h)
    logits = (2.0 * torch.randn(n, C, h, w, generator=g)).cuda().requires_grad_(True)
    labels = make_labels(n, H, W, C, 0.1, 8 + h).cuda()
    want = to.hard_cross_entropy(to.upsample_bilinear_ac(logits, (H, W)).div(T), labels)
    want_g, = torch.autograd.grad(want, logits)
    from rnd_semantic_segmentation_b200 import ops
    x2 = logits.detach().clone().requires_grad_(True)
    loss = ops.upsample_cross_entropy(x2, labels, 255, T)
    (0.5 * loss).backward()
    assert abs(loss.item() - want.item()) <= TOL * abs(want.item())
    assert rel_err(x2.grad, 0.5 * want_g) <= TOL
    # deterministic: a second run is bit-identical
    x3 = logits.detach().clone().requires_grad_(True)
    l3 = ops.upsample_cross_entropy(x3, labels, 255, T)
    (0.5 * l3).backward()
    assert torch.equal(l3, loss) and torch.equal(x3.grad, x2.grad)


def test_k2_all_ignored_is_nan_like_reference(lib):
    from rnd_semantic_segmentation_b200 import ops
    logits = torch.randn(1, 5, 7, 7, device="cuda")
    labels = torch.full((1, 20, 20), 255, dtype=torch.int64, device="cuda")
    assert torch.isnan(ops.upsample_cross_entropy(logits, labels))


# ------------------------------------------------------------------ K3
@pytest.mark.parametrize("n,K,H,W,weighted", [(2, 38, 64, 96, False), (1, 38, 33, 47, True), (2, 4, 50, 50, False), (1, 60, 17, 19, True),
                                             (4, 38, 128, 256, False)])
def test_k3_soft_label_ce(lib, n, K, H, W, weighted):
    g = torch.Generator().manual_seed(11 + K)
    pred = (3 * torch.randn(n, K, H, W, generator=g)).cuda().requires_grad_(True)
    soft = torch.softmax(2 * torch.randn(n, K, H, W, generator=g), 1).cuda()
    soft[:, K // 2:] = 0
    wts = torch.rand(n, H, W, generator=g).cuda() if weighted else None
    want = to.soft_label_cross_entropy(pred, soft, wts)
    want_g, = torch.autograd.grad(0.001 * want, pred)
    from rnd_semantic_segmentation_b200 import soft_label_cross_entropy
    p2 = pred.detach().clone().requires_grad_(True)
    loss = soft_label_cross_entropy(p2, soft, wts)
    (0.001 * loss).backward()
    assert abs(loss.item() - want.item()) <= TOL * abs(want.item())
    assert rel_err(p2.grad, want_g) <= TOL


# ------------------------------------------------------------------ K5 (fused FADA discriminator loss tail)
@pytest.mark.parametrize("n,C,h,w,H,W,slot", [(2, 19, 33, 65, 264, 520, 0), (1, 19, 64, 128, 512, 1024, 1), (2, 2, 44, 44, 352, 352, 1),
                                             (1, 7, 9, 11, 50, 70, 0), (1, 19, 17, 23, 100, 131, 1), (1, 24, 8, 8, 40, 40, 0), (1, 30, 8, 8, 40, 40, 1),
                                             (2, 11, 16, 32, 128, 256, 1)])
def test_k5_fada_soft_label_loss(lib, n, C, h, w, H, W, slot):
    import rnd_semantic_segmentation_b200 as b200
    g = torch.Generator().manual_seed(31 + C + h)
    d = (1.5 * torch.randn(n, 2 * C, h, w, generator=g)).cuda().requires_grad_(True)
    seg = (4.0 * torch.randn(n, C, h, w, generator=g)).cuda()
    # oracle: the reference sequence on materialised full-resolution tensors (aspp_fada.py:93-124)
    up_d = to.upsample_bilinear_ac(d, (H, W))
    q = to.build_soft_label(to.upsample_bilinear_ac(seg, (H, W)).div(1.8), slot)
    want = to.soft_label_cross_entropy(up_d, q)
    want_g, = torch.autograd.grad(0.5 * want, d)
    d2 = d.detach().clone().requires_grad_(True)
    loss = b200.fada_soft_label_loss(d2, seg, (H, W), slot)
    (0.5 * loss).backward()
    assert abs(loss.item() - want.item()) <= TOL * abs(want.item())
    assert rel_err(d2.grad, want_g) <= TOL
    d3 = d.detach().clone().requires_grad_(True)
    l3 = b200.fada_soft_label_loss(d3, seg, (H, W), slot)
    (0.5 * l3).backward()
    assert torch.equal(l3, loss) and torch.equal(d3.grad, d2.grad)        # deterministic


@pytest.mark.parametrize("M,N,K", [(128, 148 * 224, 64), (640, 148 * 192, 128), (100, 148 * 224 - 52, 96), (640, 32768, 192)])
@pytest.mark.parametrize("share", [0, 2])
def test_gemm_core_narrow_tiles(lib, M, N, K, share):
    """Tile widths 224 / 192 (picked when they turn the tile count into whole rounds of the 148 SMs; the last shape is the eval
    head GEMM's: 5 x 128 tiles of 256 = 5 rounds, 5 x 147 tiles of 224 = 5 shorter rounds) against the CUDA-core reference, with and
    without 2-CTA multicast of A (odd N-tile counts leave the last pair half empty)."""
    for narrow in (True, False):
        lib.gemm_set_narrow_tiles(narrow)
        try:
            err, ref = lib.gemm_selftest(M, N, K, False, False, 1, 0, share)
        finally:
            lib.gemm_set_narrow_tiles(True)
        assert ref > 0 and err <= 1e-3 * ref, (narrow, err, ref)


# ------------------------------------------------------------------ K1
def _head_pair(cin, C, seed):
    torch.manual_seed(seed)
    ref = to.AsppHeadOracle(cin, RATES, RATES, C)
    from rnd_semantic_segmentation_b200 import ASPP_Classifier_V2
    torch.manual_seed(seed)
    ours = ASPP_Classifier_V2(cin, RATES, RATES, C)
    for (ka, va), (kb, vb) in zip(ref.state_dict().items(), ours.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)          # same seed -> same init order -> identical parameters
    return ref, ours.cuda()


@pytest.mark.parametrize("n,cin,C,h,w", [(2, 2048, 19, 33, 65), (1, 256, 19, 64, 128), (3, 128, 2, 44, 44), (1, 64, 7, 9, 11), (2, 1024, 19, 17, 23)])
def test_k1_head_forward_backward(lib, n, cin, C, h, w):
    ref, ours = _head_pair(cin, C, seed=20 + C)
    g = torch.Generator().manual_seed(21 + h)
    x = torch.relu(torch.randn(n, cin, h, w, generator=g))
    go = torch.randn(n, C, h, w, generator=g) * 1e-4
    # oracle fed the same bf16-rounded operands (fp32 math on the CPU) -- the parity definition of BASELINE.md
    eff = effective_bf16_head(ref).double()
    xr = bf16_round(x).double().requires_grad_(True)
    want = eff(xr)
    xc = x.cuda().requires_grad_(True)
    got = ours(xc)
    assert rel_err(got, want) <= TOL
    print("fwd rel err vs bf16-operand oracle:", rel_err(got, want), " vs un-rounded fp32 oracle:", rel_err(got, ref(x)))
    # backward: oracle with bf16-rounded grad_output too (the GEMM operand), reported also un-rounded
    gor = bf16_round(go).double()
    want.backward(gor)
    got.backward(go.cuda())
    assert rel_err(xc.grad, xr.grad) <= TOL
    centre_w = sum(m.weight.grad[:, :, 1, 1] for m in eff.conv2d_list)   # eff carries the centre tap on branch 0 only
    for i, (m_ref, m_ours) in enumerate(zip(eff.conv2d_list, ours.conv2d_list)):
        wg = m_ref.weight.grad.clone()
        wg[:, :, 1, 1] = eff.conv2d_list[0].weight.grad[:, :, 1, 1]      # d/dW_r(centre) is the same for every branch
        assert rel_err(m_ours.weight.grad, wg) <= TOL, f"branch {i}"
        assert rel_err(m_ours.bias.grad, go.double().sum((0, 2, 3))) <= 1e-5      # bias grad is summed from the fp32 gradient


@pytest.mark.parametrize("n,cin,C,h,w,H,W", [(2, 256, 19, 16, 32, 128, 256), (1, 2048, 19, 33, 65, 264, 520), (2, 128, 2, 44, 44, 352, 352)])
def test_seam_format_bf16_channels_last(lib, n, cin, C, h, w, H, W):
    """SURVEY 8f rank 2: bf16 channels_last features in (zero-copy operand), bf16 channels_last gradient out (written by the
    dgrad GEMM's bf16 epilogue).  Same loss / weight gradients as the fp32 NCHW contract fed the same bf16-rounded features;
    the feature gradient equals the fp32 one rounded to bf16 (tolerance: one bf16 ulp of the largest entry, 2^-8 relative)."""
    from rnd_semantic_segmentation_b200 import ASPP_Classifier_V2
    torch.manual_seed(5)
    head = ASPP_Classifier_V2(cin, RATES, RATES, C).cuda()
    g = torch.Generator().manual_seed(6)
    x = bf16_round(torch.relu(torch.randn(n, cin, h, w, generator=g)))
    labels = make_labels(n, H, W, C, 0.1, 7).cuda()
    xa = x.cuda().requires_grad_(True)                                         # reference contract: fp32 NCHW
    la, _ = head.forward_loss(xa, labels)
    la.backward()
    want_w = [p.grad.clone() for p in head.parameters()]
    for p in head.parameters():
        p.grad = None
    xb = x.cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    lb, _ = head.forward_loss(xb, labels)
    lb.backward()
    assert xb.grad.dtype == torch.bfloat16 and xb.grad.shape == xb.shape
    assert xb.grad.is_contiguous(memory_format=torch.channels_last)
    assert abs(la.item() - lb.item()) <= 1e-6 * abs(la.item())
    assert rel_err(xb.grad, xa.grad) <= 2.0 ** -8
    for p, wgrad in zip(head.parameters(), want_w):
        assert rel_err(p.grad, wgrad) <= 1e-6


def test_head_grad_bucket_matches_autograd(lib):
    """distributed.HeadGradBucket: gradients written straight into the flat bucket (and all-reduced from a side stream when
    a process group exists) are bit-identical to the ones autograd returns without a bucket."""
    from rnd_semantic_segmentation_b200 import ASPP_Classifier_V2, distributed as D
    torch.manual_seed(9)
    head = ASPP_Classifier_V2(256, RATES, RATES, 19).cuda()
    g = torch.Generator().manual_seed(10)
    x = torch.relu(torch.randn(2, 256, 16, 32, generator=g)).cuda()
    labels = make_labels(2, 128, 256, 19, 0.1, 11).cuda()
    xa = x.clone().requires_grad_(True)
    la, _ = head.forward_loss(xa, labels)
    la.backward()
    want = {k: p.grad.clone() for k, p in head.named_parameters()}
    for p in head.parameters():
        p.grad = None
    bucket = D.HeadGradBucket(head)
    for step in range(2):                                  # second step: gradients are overwritten, not accumulated
        xb = x.clone().requires_grad_(True)
        lb, _ = head.forward_loss(xb, labels, grad_bucket=bucket)
        lb.backward()
        bucket.wait()
        assert torch.equal(xb.grad, xa.grad)
        for k, p in head.named_parameters():
            assert p.grad is not None and torch.equal(p.grad, want[k]), k
            assert p.grad.data_ptr() >= bucket.flat.data_ptr() and p.grad.data_ptr() < bucket.flat.data_ptr() + bucket.flat.numel() * 4


@pytest.mark.parametrize("name", ["head_c19", "head_c2", "head_c19_T18"])
def test_k1_k2_against_reference_golden(lib, golden, name):
    """End to end (head -> fused upsample+CE -> backward) against fixtures produced by the reference's own code.
    Un-rounded fp32 reference vs bf16-operand CUDA path: reported, bar 5e-3 (bf16 operand rounding, SURVEY 7.2 H3)."""
    g = golden(name)
    from rnd_semantic_segmentation_b200 import ASPP_Classifier_V2
    C = int(g["num_classes"])
    x = torch.from_numpy(g["x"]).cuda().requires_grad_(True)
    labels = torch.from_numpy(g["labels"]).cuda()
    head = ASPP_Classifier_V2(x.shape[1], RATES, RATES, C)
    head.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")})
    head.cuda()
    loss, logits_lr = head.forward_loss(x, labels, 255, float(g["temperature"]))
    loss.backward()
    assert rel_err(logits_lr, torch.from_numpy(g["logits_lr"])) <= 5e-3
    assert abs(loss.item() - float(g["loss"])) <= 5e-3 * float(g["loss"])
    assert rel_err(x.grad, torch.from_numpy(g["grad_x"])) <= 1e-2
    for k, p in head.named_parameters():
        assert rel_err(p.grad, torch.from_numpy(g["grad." + k])) <= 1e-2, k
    # the materialising API path gives the same loss
    out = head(x.detach(), labels.shape[-2:])
    l2 = F.cross_entropy(out / float(g["temperature"]), labels, ignore_index=255)
    assert abs(l2.item() - loss.item()) <= 1e-4 * abs(loss.item())


def test_eval_dropin_against_reference_golden(lib, golden):
    """inference -> .max(1)[1] -> confusion_matrix -> intersectionAndUnionGPU -> AverageMeter, as aspp_tester.py:57-74
    drives them, against the fixture the reference's own functions produced."""
    import types
    import rnd_semantic_segmentation_b200 as b200
    g = golden("eval")
    C = int(g["num_classes"])
    cfg = types.SimpleNamespace(MODEL=types.SimpleNamespace(NUM_CLASSES=C, NAME="deeplab_resnet101"))
    # logits come from the golden (fp32 reference head) so the argmax / counting path is tested bit-exactly
    meter = b200.AverageMeter()
    cmt = torch.zeros(C, C, dtype=torch.int64)

    class FixedHead(torch.nn.Module):
        def forward(self, feats, size=None):
            return feats

    for f in range(3):
        logits = torch.from_numpy(g[f"f{f}.logits_lr"]).cuda()
        y = torch.from_numpy(g[f"f{f}.y"]).cuda()
        out = b200.inference(torch.nn.Identity(), FixedHead(), logits, y, flip=False)
        pred = out.max(1)[1]
        assert torch.equal(pred.cpu(), torch.from_numpy(g[f"f{f}.pred"]))
        cm = b200.confusion_matrix(cfg, torch.flatten(pred), torch.flatten(y))
        assert torch.equal(cm, torch.from_numpy(g[f"f{f}.cm"]))
        i, u, t, r = b200.intersectionAndUnionGPU(pred, y, C, 255)
        for got, key in ((i, "I"), (u, "U"), (t, "T"), (r, "R")):
            assert got.dtype == torch.float32 and got.is_cuda
            np.testing.assert_array_equal(got.cpu().numpy(), g[f"f{f}.{key}"])
        assert bool((pred[y == 255] == 255).all())                   # the reference mutates `output` in place
        meter.update(i.cpu().numpy(), u.cpu().numpy(), t.cpu().numpy(), r.cpu().numpy())
        cmt = cmt + cm
    assert torch.equal(cmt, torch.from_numpy(g["cmt"]))
    np.testing.assert_allclose(meter.iou_sum, g["meter_iou_sum"], rtol=1e-6)
    np.testing.assert_allclose(meter.f1_sum, g["meter_f1_sum"], rtol=1e-6)


# ------------------------------------------------------------------ K6: 3x3 conv layers as tcgen05 implicit GEMMs
def _nhwc_bf16(t):
    return t.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).cuda()


def _nchw(t_nhwc, C=None):
    t = t_nhwc.float().cpu().permute(0, 3, 1, 2)
    return t if C is None else t[:, :C]


@pytest.mark.parametrize("n,ci,co,h,w,dil", [
    (2, 128, 256, 64, 128, 1),     # one 1 x 128 rectangle per image row, exact tiles
    (1, 256, 128, 33, 65, 1),      # ragged 8 x 16 rectangles, half-empty N tile
    (2, 64, 40, 9, 11, 1),         # tiny image, Co = 40 (the 2C = 38 -> 40 class of the cls layer)
    (1, 24, 16, 20, 27, 1),        # Ci < one 64-channel k-block (TMA zero-fills the rest)
    (1, 192, 64, 17, 40, 2),       # dilation 2 (padding 2)
])
def test_conv3x3_layer_forward_dgrad_wgrad(lib, n, ci, co, h, w, dil):
    g = torch.Generator().manual_seed(100 + h + ci)
    x = bf16_round(torch.randn(n, ci, h, w, generator=g))
    wt = bf16_round(torch.randn(co, ci, 3, 3, generator=g) * 0.05)
    b = torch.randn(co, generator=g) * 0.1
    go = bf16_round(torch.randn(n, co, h, w, generator=g))
    xd, wd = x.double().requires_grad_(True), wt.double().requires_grad_(True)
    z = F.conv2d(xd, wd, b.double(), padding=dil, dilation=dil)
    gx_want, gw_want = torch.autograd.grad(z, (xd, wd), go.double())
    Wf, Wb = lib.conv3x3_pack_weights([wt.cuda()])
    xq, gq = _nhwc_bf16(x), _nhwc_bf16(go)
    # forward: fp32 NCHW (exact up to accumulation order) and bf16 NHWC with the fused LeakyReLU (one bf16 rounding)
    out_f = lib.conv3x3_forward(xq, Wf, b.cuda(), None, dilation=dil, out_f32_nchw=True)
    assert rel_err(out_f, z) <= TOL
    out_b = lib.conv3x3_forward(xq, Wf, b.cuda(), 0.2, dilation=dil)
    assert rel_err(_nchw(out_b), F.leaky_relu(z, 0.2)) <= 2.0 ** -8
    assert rel_err(_nchw(lib.conv3x3_forward(xq, Wf, None, None, dilation=dil)), z - b.double().view(1, -1, 1, 1)) <= 2.0 ** -8
    # data gradient: fp32 NCHW, and bf16 NHWC with the LeakyReLU' mask of a saved activation
    assert rel_err(lib.conv3x3_dgrad(gq, Wb, dilation=dil, out_f32_nchw=True), gx_want) <= TOL
    mask_src = torch.randn(n, ci, h, w, generator=g)
    mask_src[0, 0, 0, :3] = 0.0                                     # LeakyReLU'(0) = slope
    got = lib.conv3x3_dgrad(gq, Wb, mask=_nhwc_bf16(mask_src), slope=0.2, dilation=dil)
    assert rel_err(_nchw(got), gx_want * torch.where(bf16_round(mask_src) > 0, 1.0, 0.2)) <= 2.0 ** -8
    if ci % 8 == 0:
        # the same launch with the bias gradient of the layer below folded into the epilogue: identical tensor, and column sums
        # equal to a separate pass over what was stored (both in pair mode and with one CTA per tile)
        for pair in (1, 0):
            lib.conv_set_pair(pair)
            try:
                got2, cs = lib.conv3x3_dgrad(gq, Wb, mask=_nhwc_bf16(mask_src), slope=0.2, dilation=dil, want_colsum=True)
                got_ref = lib.conv3x3_dgrad(gq, Wb, mask=_nhwc_bf16(mask_src), slope=0.2, dilation=dil)
            finally:
                lib.conv_set_pair(True)
            assert torch.equal(got2, got_ref)
            assert rel_err(cs, got2.double().sum((0, 1, 2))) <= 1e-5, f"pair={pair}"
            cs2 = lib.conv3x3_dgrad(gq, Wb, mask=_nhwc_bf16(mask_src), slope=0.2, dilation=dil, want_colsum=True)[1]
            assert torch.equal(cs, cs2)                             # deterministic
    # weight gradient (split-K chosen by the library, and forced to 1 / 3 splits); bias gradient
    for splits in (0, 1, 3):
        gw, = lib.conv3x3_wgrad(gq, xq, [co], dilation=dil, splits=splits)
        assert rel_err(gw, gw_want) <= TOL, f"splits={splits}"
    assert rel_err(lib.nhwc_bf16_colsum(gq), go.double().sum((0, 2, 3))) <= 1e-5
    a, bb = lib.nhwc_bf16_colsum(gq), lib.nhwc_bf16_colsum(gq)
    assert torch.equal(a, bb)                                       # deterministic


def test_conv3x3_concatenated_parts_and_nchw_pack(lib):
    """cls1 | cls2 as one layer: two [C,Ci,3,3] tensors packed side by side, 2C = 38 padded to 40 in the gradient operand."""
    g = torch.Generator().manual_seed(7)
    C, ci, n, h, w = 19, 128, 2, 12, 20
    w1, w2 = (bf16_round(torch.randn(C, ci, 3, 3, generator=g) * 0.05) for _ in range(2))
    x = bf16_round(torch.randn(n, ci, h, w, generator=g))
    go = torch.randn(n, 2 * C, h, w, generator=g)
    Wf, Wb = lib.conv3x3_pack_weights([w1.cuda(), w2.cuda()])
    assert tuple(Wf.shape) == (9, 38, ci) and tuple(Wb.shape) == (9, ci, 40)
    xd = x.double().requires_grad_(True)
    wd = [t.double().requires_grad_(True) for t in (w1, w2)]
    z = torch.cat([F.conv2d(xd, t, padding=1) for t in wd], 1)
    out = lib.conv3x3_forward(_nhwc_bf16(x), Wf, None, None, out_f32_nchw=True)
    assert rel_err(out, z) <= TOL
    G = lib.nchw_to_nhwc_bf16(go.cuda())
    assert tuple(G.shape) == (n, h, w, 40) and float(G[..., 38:].abs().max()) == 0.0
    assert torch.equal(_nchw(G, 38), bf16_round(go))
    gx_want, g1_want, g2_want = torch.autograd.grad(z, (xd, *wd), bf16_round(go).double())
    assert rel_err(lib.conv3x3_dgrad(G, Wb, out_f32_nchw=True), gx_want) <= TOL
    g1, g2 = lib.conv3x3_wgrad(G, _nhwc_bf16(x), [C, C])
    assert rel_err(g1, g1_want) <= TOL and rel_err(g2, g2_want) <= TOL
    assert rel_err(lib.nhwc_bf16_colsum(G, 38), bf16_round(go).double().sum((0, 2, 3))) <= 1e-5


@pytest.mark.parametrize("n,cin,ndf,C,h,w", [(2, 256, 64, 19, 33, 65), (1, 2048, 256, 19, 32, 64), (2, 64, 32, 2, 44, 44), (1, 24, 16, 3, 20, 27)])
def test_discriminator_stack_forward_backward(lib, n, cin, ndf, C, h, w):
    """PixelDiscriminator.logits / backward (tcgen05 conv stack) against the oracle module applying the same bf16 roundings.
    Every single layer meets 1e-3 (test_conv3x3_layer_*).  Through the CHAIN the bar is 3e-3: an fp32-vs-fp64 accumulation
    difference of ~1e-6 relative flips the bf16 rounding of about one stored activation in a thousand by one ulp (2^-8), and
    those flips propagate through the next layers -- the floor of any comparison across bf16-stored activations."""
    STACK_TOL = 3e-3
    import copy
    import rnd_semantic_segmentation_b200 as b200
    from helpers import discriminator_bf16_oracle
    torch.manual_seed(40 + C)
    ref = to.PixelDiscriminatorOracle(cin, ndf, num_classes=C)
    torch.manual_seed(40 + C)
    ours = b200.PixelDiscriminator(cin, ndf, num_classes=C)
    for (ka, va), (kb, vb) in zip(ref.state_dict().items(), ours.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)
    ours.cuda()
    g = torch.Generator().manual_seed(41 + h)
    x = torch.relu(torch.randn(n, cin, h, w, generator=g))
    go = torch.randn(n, 2 * C, h, w, generator=g) * 1e-3
    xc = x.cuda().requires_grad_(True)
    got = ours(xc)
    assert tuple(got.shape) == (n, 2 * C, h, w)
    # INDEPENDENT oracle: its LeakyReLU branches follow its OWN fp64 pre-activations (no mask is taken from the CUDA path).
    # The CUDA stack derives the backward slope from the sign of its stored bf16 activation; the two can only disagree where a
    # pre-activation lies within fp32-accumulation distance (~1e-6 relative) of zero.  Count those disagreements against the
    # activations the CUDA layers store, and bound them: measured 0 for the small stacks and 20 of 786 432 (2.5e-5) for the
    # 2048-channel one (fp32 accumulation over K = 18 432, and layer 2 sees layer-1 activations that differ by single bf16 ulps).
    refd = copy.deepcopy(ref).double()
    xr = x.double().requires_grad_(True)
    want = discriminator_bf16_oracle(refd, xr, None)
    with torch.no_grad():
        (Wf1, _), (Wf2, _), _, _ = ours._packed_weights()
        A1 = lib.conv3x3_forward(_nhwc_bf16(x), Wf1, ours.D[0].bias.detach(), 0.2)
        A2 = lib.conv3x3_forward(A1, Wf2, ours.D[2].bias.detach(), 0.2)
        r = lambda t: bf16_round(t.float()).double()  # noqa: E731
        z1 = F.conv2d(r(x.double()), r(refd.D[0].weight), refd.D[0].bias, padding=1)
        a1 = r(F.leaky_relu(z1, 0.2))
        z2 = F.conv2d(a1, r(refd.D[2].weight), refd.D[2].bias, padding=1)
        flips = int(((_nchw(A1) > 0) != (z1 > 0)).sum()) + int(((_nchw(A2) > 0) != (z2 > 0)).sum())
        n_act = z1.numel() + z2.numel()
    print(f"LeakyReLU sign disagreements CUDA vs independent fp64 oracle: {flips} of {n_act} pre-activations")
    assert flips <= max(2, int(1e-4 * n_act)), (flips, n_act)
    assert rel_err(got, want) <= STACK_TOL
    print("D logits rel err vs same-rounding oracle:", rel_err(got, want), " vs fp32 reference module:", rel_err(got, ref(x)))
    assert rel_err(got, ref(x)) <= 2e-2
    want.backward(go.double())
    got.backward(go.cuda())
    # with no sign disagreement the un-masked comparison holds at the chain tolerance; each disagreement changes one element of
    # an inter-layer gradient by the slope ratio, so then the bound is stated in L2
    # (k disagreements among n activations move the L2 norm of an inter-layer gradient by about 0.8 * sqrt(k / n): 4e-3 here)
    grad_ok = (lambda a, b: rel_err(a, b) <= STACK_TOL) if flips == 0 else \
        (lambda a, b: ((a.detach().double().cpu() - b.double()).norm() / b.double().norm()).item() <= 2.5 * (flips / n_act) ** 0.5 + STACK_TOL)
    assert grad_ok(xc.grad, xr.grad)
    for (name, p_ref), (_, p_ours) in zip(refd.named_parameters(), ours.named_parameters()):
        assert grad_ok(p_ours.grad, p_ref.grad), name
    # weights-only backward (the discriminator's own update on detached features, aspp_fada.py:119-125) and determinism
    ours.zero_grad()
    out2 = ours(x.cuda())
    out2.backward(go.cuda())
    g_first = [p.grad.clone() for p in ours.parameters()]
    for p_ours, (name, p_ref) in zip(ours.parameters(), refd.named_parameters()):
        assert grad_ok(p_ours.grad, p_ref.grad), name
    ours.zero_grad()
    ours(x.cuda()).backward(go.cuda())
    assert all(torch.equal(a, p.grad) for a, p in zip(g_first, ours.parameters()))


def test_conv3x3_full_size_adversarial_layer1(lib):
    """BASELINE configs[2] at full size (4 x 2048 x 64 x 128 -> 256): forward, data gradient and weight gradient of the dominant
    layer against torch's strict-fp32 convolution on the GPU, fed the same bf16-rounded operands; both tile modes (one CTA per
    tile, CTA pairs on tcgen05.mma.cta_group::2) must agree with it and give bit-identical results run to run."""
    g = torch.Generator(device="cuda").manual_seed(5)
    n, ci, co, h, w = 4, 2048, 256, 64, 128
    x = bf16_round(torch.relu(torch.randn(n, ci, h, w, device="cuda", generator=g)))
    wt = bf16_round(torch.randn(co, ci, 3, 3, device="cuda", generator=g) * 0.01)
    go = bf16_round(torch.randn(n, co, h, w, device="cuda", generator=g) * 1e-3)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        xr, wr = x.clone().requires_grad_(True), wt.clone().requires_grad_(True)
        z = F.conv2d(xr, wr, padding=1)
        gx_want, gw_want = torch.autograd.grad(z, (xr, wr), go)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    Wf, Wb = lib.conv3x3_pack_weights([wt])
    xq = x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    gq = go.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    outs = {}
    for pair in (False, True):
        lib.conv_set_pair(pair)
        try:
            out = lib.conv3x3_forward(xq, Wf, None, None, out_f32_nchw=True)
            gx = lib.conv3x3_dgrad(gq, Wb, out_f32_nchw=True)
            gw, = lib.conv3x3_wgrad(gq, xq, [co])
            assert torch.equal(out, lib.conv3x3_forward(xq, Wf, None, None, out_f32_nchw=True))
            assert torch.equal(gw, lib.conv3x3_wgrad(gq, xq, [co])[0])
        finally:
            lib.conv_set_pair(True)
        assert rel_err(out, z) <= TOL and rel_err(gx, gx_want) <= TOL and rel_err(gw, gw_want) <= TOL, f"pair={pair}"
        outs[pair] = (out, gx, gw)
    # both modes accumulate each output in the same k order: identical bits
    assert all(torch.equal(a, b) for a, b in zip(outs[False], outs[True]))


def test_fada_iteration_losses_match_oracle(lib):
    """The whole adversarial iteration after the backbone (aspp_fada.py:91-125) through the fused entry points -- head
    forward_loss, head logits, three discriminator passes with forward_soft_loss -- against oracle.fada_step: the four losses
    the reference logs, and the gradients left on the parameters and on the target features."""
    import rnd_semantic_segmentation_b200 as b200
    n, cin, C, h, w, H, W = 2, 256, 19, 16, 32, 128, 256
    torch.manual_seed(77)
    ref_head = to.AsppHeadOracle(cin, RATES, RATES, C)
    ref_D = to.PixelDiscriminatorOracle(cin, 64, num_classes=C)
    head = b200.ASPP_Classifier_V2(cin, RATES, RATES, C)
    head.load_state_dict(ref_head.state_dict())
    D = b200.PixelDiscriminator(cin, 64, num_classes=C)
    D.load_state_dict(ref_D.state_dict())
    head.cuda(), D.cuda()
    g = torch.Generator().manual_seed(78)
    src, tgt = (torch.relu(torch.randn(n, cin, h, w, generator=g)) for _ in range(2))
    lab = make_labels(n, H, W, C, 0.1, 79)
    want = to.fada_step(ref_head, ref_D, src, tgt, lab)
    size = (H, W)
    src_fea, tgt_fea = src.cuda().requires_grad_(True), tgt.cuda().requires_grad_(True)
    loss_seg, src_lr = head.forward_loss(src_fea, lab.cuda(), temperature=1.8)
    loss_seg.backward()
    with torch.no_grad():
        tgt_lr = head.logits(tgt_fea)
    loss_adv = 0.001 * D.forward_soft_loss(tgt_fea, tgt_lr, size, slot=0)
    loss_adv.backward()
    D.zero_grad()
    loss_d_src = 0.5 * D.forward_soft_loss(src_fea.detach(), src_lr, size, slot=0)
    loss_d_src.backward()
    loss_d_tgt = 0.5 * D.forward_soft_loss(tgt_fea.detach(), tgt_lr, size, slot=1)
    loss_d_tgt.backward()
    for name, got, exp in zip(("seg", "adv_tgt", "D_src", "D_tgt"), (loss_seg, loss_adv, loss_d_src, loss_d_tgt), want):
        assert abs(got.item() - exp.item()) <= 5e-3 * abs(exp.item()), (name, got.item(), exp.item())
    # bf16 operands / stored activations vs the UN-ROUNDED fp32 oracle (the same-rounding bars are in the K1 / K6 tests):
    # head gradients to 2e-2 max-abs; discriminator gradients to 3e-2 in L2 -- with only 1024 pixels the few pre-activations
    # that take the other LeakyReLU slope after bf16 operand rounding are visible in single weight-gradient elements
    for (name, p), pr in zip(head.named_parameters(), ref_head.parameters()):
        assert rel_err(p.grad, pr.grad) <= 2e-2, name
    for (name, p), pr in zip(D.named_parameters(), ref_D.parameters()):
        got, exp = p.grad.detach().cpu().double(), pr.grad.double()
        assert ((got - exp).norm() / exp.norm()).item() <= 3e-2, name


def test_fada_iterations_with_optimizer_steps_match_oracle(lib):
    """Three consecutive adversarial iterations INCLUDING the optimizer steps where the reference takes them (aspp_fada.py:
    80-127 after the backbone: optimizer_cls.step() after the adversarial backward, optimizer_D.step() at the end, poly learning
    rates rewritten into the param groups) -- FusedSGD / FusedAdam on the gradients our kernels produce, against torch.optim on
    the oracle's: losses of every iteration, and the parameter UPDATES accumulated over the three iterations."""
    import copy
    import rnd_semantic_segmentation_b200 as b200
    n, cin, C, h, w, H, W = 2, 256, 19, 16, 32, 128, 256
    torch.manual_seed(91)
    ref_head = to.AsppHeadOracle(cin, RATES, RATES, C)
    ref_D = to.PixelDiscriminatorOracle(cin, 64, num_classes=C)
    head = b200.ASPP_Classifier_V2(cin, RATES, RATES, C)
    head.load_state_dict(ref_head.state_dict())
    D = b200.PixelDiscriminator(cin, 64, num_classes=C)
    D.load_state_dict(ref_D.state_dict())
    head.cuda(), D.cuda()
    head0, D0 = copy.deepcopy(ref_head.state_dict()), copy.deepcopy(ref_D.state_dict())
    base_lr, base_lr_d, max_iter = 2.5e-4, 1e-4, 10
    ref_cls = torch.optim.SGD(ref_head.parameters(), lr=base_lr * 10, momentum=0.9, weight_decay=5e-4)       # aspp_trainer.py:26
    ref_opt_d = torch.optim.Adam(ref_D.parameters(), lr=base_lr_d, betas=(0.9, 0.99))                        # fada_adapter.py:24
    opt_cls = b200.FusedSGD(head.parameters(), lr=base_lr * 10, momentum=0.9, weight_decay=5e-4)
    opt_d = b200.FusedAdam(D.parameters(), lr=base_lr_d, betas=(0.9, 0.99))
    g = torch.Generator().manual_seed(92)
    size = (H, W)
    for it in range(3):
        src, tgt = (torch.relu(torch.randn(n, cin, h, w, generator=g)) for _ in range(2))
        lab = make_labels(n, H, W, C, 0.1, 93 + it)
        lr = b200.adjust_learning_rate('poly', base_lr, it, max_iter, 0.9)
        lr_d = b200.adjust_learning_rate('poly', base_lr_d, it, max_iter, 0.9)
        for o in (ref_cls, opt_cls):
            for grp in o.param_groups:
                grp['lr'] = lr * 10
        for o in (ref_opt_d, opt_d):
            for grp in o.param_groups:
                grp['lr'] = lr_d
        want = to.fada_iteration(ref_head, ref_D, ref_cls, ref_opt_d, src, tgt, lab)
        opt_cls.zero_grad()
        opt_d.zero_grad()
        src_fea, tgt_fea = src.cuda().requires_grad_(True), tgt.cuda().requires_grad_(True)
        loss_seg, src_lr = head.forward_loss(src_fea, lab.cuda(), temperature=1.8)
        loss_seg.backward()
        with torch.no_grad():
            tgt_lr = head.logits(tgt_fea)
        loss_adv = 0.001 * D.forward_soft_loss(tgt_fea, tgt_lr, size, slot=0)
        loss_adv.backward()
        opt_cls.step()
        opt_d.zero_grad()
        loss_d_src = 0.5 * D.forward_soft_loss(src_fea.detach(), src_lr, size, slot=0)
        loss_d_src.backward()
        loss_d_tgt = 0.5 * D.forward_soft_loss(tgt_fea.detach(), tgt_lr, size, slot=1)
        loss_d_tgt.backward()
        opt_d.step()
        for name, got, exp in zip(("seg", "adv_tgt", "D_src", "D_tgt"), (loss_seg, loss_adv, loss_d_src, loss_d_tgt), want):
            assert abs(got.item() - exp.item()) <= 5e-3 * abs(exp.item()), (it, name, got.item(), exp.item())
    # updates (parameter minus its initial value): SGD's follow the gradients (bf16-operand tolerance of the K1 tests, 2e-2);
    # Adam's are lr * m / sqrt(v) ~ lr * sign-like, so elements whose gradient is near zero amplify any gradient difference:
    # compare those in L2
    for (name, p), pr in zip(head.named_parameters(), ref_head.parameters()):
        d_got, d_exp = p.detach().cpu().double() - head0[name].double(), pr.detach().double() - head0[name].double()
        assert float(d_exp.abs().max()) > 0 and rel_err(d_got, d_exp) <= 2e-2, name
    for (name, p), pr in zip(D.named_parameters(), ref_D.parameters()):
        d_got, d_exp = p.detach().cpu().double() - D0[name].double(), pr.detach().double() - D0[name].double()
        assert float(d_exp.norm()) > 0 and ((d_got - d_exp).norm() / d_exp.norm()).item() <= 0.1, name
    assert float(opt_d.state[next(iter(D.parameters()))]["step"]) == 3


def test_cuda_graph_capture_train_eval_and_discriminator(lib):
    """SURVEY 8b: the ops are capture-safe.  One train step (head forward_loss + backward), one eval step (head logits + fused
    argmax / confusion) and one discriminator loss step are captured in CUDA graphs; after the inputs are overwritten in place the
    replays must give exactly what the eager calls give on the new inputs."""
    import rnd_semantic_segmentation_b200 as b200
    from rnd_semantic_segmentation_b200 import synth
    C, cin, h, w, H, W = 19, 256, 16, 32, 128, 256
    torch.manual_seed(11)
    head = synth.scale_head_for_unit_logits(b200.ASPP_Classifier_V2(cin, RATES, RATES, C), 5.0).cuda()
    D = b200.PixelDiscriminator(cin, 64, num_classes=C).cuda()
    params = list(head.parameters()) + list(D.parameters())
    gen = torch.Generator().manual_seed(12)
    xs = [torch.relu(torch.randn(2, cin, h, w, generator=gen)).cuda() for _ in range(2)]
    ys = [make_labels(2, H, W, C, 0.1, 13 + i).cuda() for i in range(2)]
    x, y = xs[0].clone(), ys[0].clone()
    cm = torch.zeros(C, C, dtype=torch.int64, device="cuda")
    b200.set_feature_pack_cache(0)
    try:
        def step(x_in, y_in, cm_in):
            for p in params:
                p.grad = None
            xg = x_in.detach().requires_grad_(True)
            loss, lg = head.forward_loss(xg, y_in)
            loss.backward()
            b200.segmentation_eval_step(lg, y_in, cm=cm_in)
            xd = x_in.detach().requires_grad_(True)
            loss_d = D.forward_soft_loss(xd, lg, (H, W), slot=1)
            loss_d.backward()
            return loss, xg.grad, loss_d, xd.grad

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                     # warm-up: lazy kernel attributes, packed weights, scratch
            for _ in range(3):
                step(x, y, cm)
        torch.cuda.current_stream().wait_stream(side)
        for p in params:
            p.grad = None
        cm.zero_()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            outs = step(x, y, cm)
            grads = [p.grad for p in params]
        for i in (1, 0, 1):
            x.copy_(xs[i]); y.copy_(ys[i]); cm.zero_()
            graph.replay()
            torch.cuda.synchronize()
            got = [t.clone() for t in outs] + [g.clone() for g in grads] + [cm.clone()]
            cm_e = torch.zeros_like(cm)
            want = list(step(xs[i], ys[i], cm_e)) + [p.grad for p in params] + [cm_e]
            for a, b in zip(got, want):
                assert torch.equal(a, b)
    finally:
        b200.set_feature_pack_cache(0)


def test_discriminator_tail_and_soft_ce_golden(lib, golden):
    import rnd_semantic_segmentation_b200 as b200
    g = golden("discriminator")
    C = int(g["num_classes"])
    D = b200.PixelDiscriminator(24, 16, num_classes=C)
    D.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")})
    D.cuda()
    x = torch.from_numpy(g["x"]).cuda()
    out_hr = D(x, (20, 27))
    # tcgen05 conv stack with bf16 operands / activations against the reference's fp32 fixture: the bf16 rounding of three
    # chained layers bounds this comparison (the same-rounding oracle comparison at 1e-3 is test_discriminator_stack_*)
    print("D(x, size) rel err vs the reference's fp32 golden:", rel_err(out_hr, torch.from_numpy(g["out_hr"])))
    assert rel_err(out_hr, torch.from_numpy(g["out_hr"])) <= 1e-2
    soft = torch.from_numpy(g["soft"]).cuda()
    q0 = torch.cat((soft, torch.zeros_like(soft)), 1)
    loss = b200.soft_label_cross_entropy(out_hr, q0)
    assert abs(loss.item() - float(g["loss_slot0"])) <= 5e-3 * float(g["loss_slot0"])
    gw, = torch.autograd.grad(loss, D.cls1.weight)
    assert rel_err(gw, torch.from_numpy(g["grad_cls1_weight_slot0"])) <= 1e-2


def test_full_size_properties_config1(lib):
    """BASELINE config 1 at full size through size-independent properties: linearity of the head in x,
    sum of the CE gradient over classes is zero at every low-res logit, confusion matrix total == valid pixels."""
    from rnd_semantic_segmentation_b200 import ASPP_Classifier_V2, ops, synth
    torch.manual_seed(0)
    head = ASPP_Classifier_V2(2048, RATES, RATES, 19).cuda()
    x = synth.make_features(2, 2048, 65, 129, device="cuda")
    labels = synth.make_labels(2, 512, 1024, 19, device="cuda")
    with torch.no_grad():
        y1 = head.logits(x)
        y2 = head.logits(2 * x)
        bias = sum(m.bias for m in head.conv2d_list).view(1, -1, 1, 1)
        assert rel_err(y2 - bias, 2 * (y1 - bias)) <= 1e-5              # bf16(2x) == 2*bf16(x): exact linearity
    lg = y1.clone().requires_grad_(True)
    ops.upsample_cross_entropy(lg, labels).backward()
    assert lg.grad.sum(1).abs().max().item() <= 1e-6 * lg.grad.abs().max().item() * 19 + 1e-12
    cm, _ = ops._lib.upsample_argmax_confusion(y1, labels, (512, 1024))
    assert int(cm.sum()) == int((labels != 255).sum())


# ------------------------------------------------------------------ K7: fused test-time augmentation (SURVEY 8f rank 3)
def _tta_members(C, shapes, sigma, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(1, C, h, w, generator=g) * sigma).cuda() for h, w in shapes]


@pytest.mark.parametrize("C,shapes,flips,divisors,H,W", [
    (19, [(64, 128), (64, 128)], [False, True], (2,), 512, 1024),                       # inference(flip=True), train-crop size
    (19, [(128, 256), (128, 256)], [False, True], (2,), 1024, 2048),                    # ... at the 1024 x 2048 eval size
    (19, [(45, 90), (45, 90), (64, 128), (64, 128), (84, 167), (84, 167)], [False, True] * 3, (3, 2), 512, 1024),  # multi-scale + flip
    (19, [(23, 45), (33, 65), (43, 84)], [False] * 3, (3,), 260, 517),                  # multi-scale, no flip, odd sizes
    (2, [(44, 44), (44, 44)], [False, True], (2,), 352, 352),                           # kvasir polyp head
    (7, [(9, 11)], [True], (), 50, 70),                                                 # one mirrored member, no division
    (30, [(8, 8), (12, 10)], [False, False], (2,), 64, 61),                             # CT = 32 path
])
@pytest.mark.parametrize("sigma", [1.0, 0.01])
def test_k7_tta_bit_exact_against_torch_cuda(lib, C, shapes, flips, divisors, H, W, sigma):
    """Probabilities, argmax and confusion matrix of the fused kernel against the reference's op sequence (utility.py:179-209)
    run with torch CUDA ops on the same low-res logits: bit-exact (sigma = 0.01 puts many classes within a few ulp)."""
    members = _tta_members(C, shapes, sigma, seed=300 + C + len(shapes))
    labels = make_labels(1, H, W, C, 0.1, 17).cuda()
    want = to.tta_probabilities(members, flips, (H, W), divisors)
    want_pred = want.max(1)[1]
    cm, pred, probs = lib.tta_argmax_confusion(members, flips, (H, W), labels=labels, divisors=divisors, want_pred=True,
                                               want_probs=True)
    assert rel_err(probs.unsqueeze(0), want) <= 1e-6
    assert torch.equal(probs.unsqueeze(0), want), f"max abs diff {(probs.unsqueeze(0) - want).abs().max().item():.3e}"
    assert torch.equal(pred.unsqueeze(0), want_pred)
    assert torch.equal(cm.cpu(), to.confusion_matrix_bincount(C, want_pred.flatten().cpu(), labels.flatten().cpu()))
    # outputs are independent of each other, and the matrix accumulates
    cm2, pred2, probs2 = lib.tta_argmax_confusion(members, flips, (H, W), labels=labels, divisors=divisors, cm=cm.clone())
    assert pred2 is None and probs2 is None and torch.equal(cm2, 2 * cm)
    _, pred3, _ = lib.tta_argmax_confusion(members, flips, (H, W), divisors=divisors, want_pred=True)
    assert torch.equal(pred3, pred)


def test_k7_flip_symmetry_and_errors(lib):
    """Size-independent properties: mirroring every member and toggling every flip flag leaves the output unchanged (up to
    the rounding of the mirrored sampling positions); a member averaged
    with its own mirror image (flagged as mirrored) reproduces the single member; IEEE-division mode equals reciprocal mode for
    powers of two."""
    C, H, W = 19, 96, 160
    a, b = _tta_members(C, [(12, 20), (17, 31)], 1.0, 5)
    _, pred, probs = lib.tta_argmax_confusion([a, b], [False, True], (H, W), divisors=(2,), want_pred=True, want_probs=True)
    _, pred_m, probs_m = lib.tta_argmax_confusion([a.flip(3).contiguous(), b.flip(3).contiguous()], [True, False], (H, W),
                                                  divisors=(2,), want_pred=True, want_probs=True)
    assert rel_err(probs_m, probs) <= 1e-5 and (pred_m != pred).float().mean().item() < 1e-3
    _, _, probs_s = lib.tta_argmax_confusion([a, a.flip(3).contiguous()], [False, True], (H, W), divisors=(2,), want_probs=True)
    _, _, probs_1 = lib.tta_argmax_confusion([a], [False], (H, W), want_probs=True)
    assert rel_err(probs_s, probs_1) <= 1e-5
    assert torch.equal(probs_1.unsqueeze(0), to.eval_probabilities(a, (H, W)))             # one plain member == inference(flip=False)
    _, pred_e, probs_e = lib.tta_argmax_confusion([a, b], [False, True], (H, W), divisors=(2,), want_pred=True, want_probs=True,
                                                  div_exact=True)
    assert torch.equal(probs_e, probs) and torch.equal(pred_e, pred)
    with pytest.raises(lib.B200SegError):
        lib.tta_argmax_confusion([a] * 9, [False] * 9, (H, W), want_pred=True)
    with pytest.raises(lib.B200SegError):
        lib.tta_argmax_confusion([a, b], [False, True], (H, W), divisors=(2,))            # nothing to compute
    with pytest.raises(lib.B200SegError):
        lib.tta_argmax_confusion([a.cpu()], [False], (H, W), want_pred=True)              # no CPU fallback


def test_k7_dropin_against_reference_golden(lib, golden):
    """b200.inference(flip=True) / b200.multi_scale_inference driven like core/testers/aspp_tester.py:60-72, on the member logits
    the REFERENCE produced (tests/golden/tta.npz, CPU): probabilities to 1e-6, argmax equal wherever the top two are > 1e-6 apart."""
    import types
    import rnd_semantic_segmentation_b200 as b200
    g = golden("tta")
    C = int(g["num_classes"])
    cfg = types.SimpleNamespace(MODEL=types.SimpleNamespace(NUM_CLASSES=C, NAME="deeplab_resnet101"))
    image, label = torch.from_numpy(g["image"]).cuda(), torch.from_numpy(g["label"]).cuda()

    class Replay(torch.nn.Module):
        def __init__(self, outs):
            super().__init__()
            self.outs, self.k = outs, 0

        def forward(self, feats, size=None):
            out = self.outs[self.k]
            self.k += 1
            return out

    def check(out, name):
        want = torch.from_numpy(g[f"{name}.probs"])
        assert tuple(out.shape) == tuple(want.shape)
        pred = out.max(1)[1]
        assert tuple(pred.shape) == (1,) + tuple(label.shape[-2:]) and pred.dtype == torch.int64
        top2 = want.topk(2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-6
        assert torch.equal(pred.cpu()[clear], torch.from_numpy(g[f"{name}.pred"])[clear])
        cm = b200.confusion_matrix(cfg, torch.flatten(pred), torch.flatten(label))
        assert torch.equal(cm, to.confusion_matrix_bincount(C, pred.flatten().cpu(), label.flatten().cpu()))
        np.testing.assert_allclose(out.cpu().numpy(), want.numpy(), rtol=2e-6, atol=1e-7)      # materialises (the API-compat path)

    both = torch.cat([torch.from_numpy(g["flip.member0"]), torch.from_numpy(g["flip.member1"])], 0).cuda()
    check(b200.inference(torch.nn.Identity(), Replay([both]), image, label, flip=True), "flip")
    for name, flip in (("ms", True), ("ms_noflip", False)):
        members = [torch.from_numpy(g[f"{name}.member{k}"]).cuda() for k in range(int(g[f"{name}.n_members"]))]
        out = b200.multi_scale_inference(torch.nn.Identity(), Replay(members), image, label, flip=flip,
                                         scales=[float(s) for s in g["scales"]])
        check(out, name)


# ------------------------------------------------------------------ K8: fused optimizer steps (SURVEY 8f rank 4)
OPT_TOL = 1e-6      # relative (max-abs / max-abs): one-ulp rounding differences of single intermediates against torch.optim


def test_k8_fused_sgd_adam_against_reference_golden(lib, golden):
    """FusedSGD / FusedAdam driven exactly as aspp_trainer.py:77-81,94-95 drives torch.optim (lr rewritten in the param groups
    every iteration from the poly schedule) against the parameters and optimizer states the reference's own setup produced."""
    import rnd_semantic_segmentation_b200 as b200
    g = golden("optim")
    n, steps = int(g["n"]), int(g["steps"])

    def run(ctor, scale):
        ps = [torch.nn.Parameter(torch.from_numpy(g[f"p0.{i}"]).cuda()) for i in range(n)]
        opt = ctor(ps)
        for k in range(steps):
            lr = b200.adjust_learning_rate('poly', float(g["base_lr"]), k, int(g["max_iter"]), float(g["power"]))
            assert lr == float(g["lrs"][k])
            for grp in opt.param_groups:
                grp['lr'] = lr * scale
            opt.zero_grad()
            for i, p in enumerate(ps):
                p.grad = torch.from_numpy(g[f"g{k}.{i}"]).cuda()
            opt.step()
        return ps, opt

    launches0 = lib.load().b200seg_launch_count()
    ps, opt = run(lambda ps: b200.FusedSGD(ps, lr=float(g["base_lr"]) * 10, momentum=0.9, weight_decay=5e-4), 10)
    assert lib.load().b200seg_launch_count() - launches0 == steps              # one launch per step for the whole group
    for i, p in enumerate(ps):
        assert rel_err(p, torch.from_numpy(g[f"sgd.p.{i}"])) <= OPT_TOL
        assert rel_err(opt.state[p]["momentum_buffer"], torch.from_numpy(g[f"sgd.buf.{i}"])) <= OPT_TOL
    ps, opt = run(lambda ps: b200.FusedAdam(ps, lr=1e-4, betas=(0.9, 0.99)), 0.4)
    for i, p in enumerate(ps):
        assert rel_err(p, torch.from_numpy(g[f"adam.p.{i}"])) <= OPT_TOL
        assert rel_err(opt.state[p]["exp_avg"], torch.from_numpy(g[f"adam.m.{i}"])) <= OPT_TOL
        assert rel_err(opt.state[p]["exp_avg_sq"], torch.from_numpy(g[f"adam.v.{i}"])) <= 4 * OPT_TOL
        assert float(opt.state[p]["step"]) == steps


@pytest.mark.parametrize("kind,hyper", [
    ("sgd", dict(lr=0.0025, momentum=0.9, weight_decay=5e-4)),
    ("sgd", dict(lr=0.01, momentum=0.9, nesterov=True)),
    ("sgd", dict(lr=0.01, momentum=0.8, dampening=0.1, weight_decay=1e-3)),
    ("sgd", dict(lr=0.05)),
    ("adam", dict(lr=1e-4, betas=(0.9, 0.99))),
    ("adam", dict(lr=1e-3, betas=(0.5, 0.999), eps=1e-6, weight_decay=1e-2)),
])
def test_k8_matches_torch_optim_and_interchanges_state(lib, kind, hyper):
    """Real parameter sets (ASPP head 8 tensors; 20 tensors = two launches), five steps against torch.optim on the GPU (both the
    single-tensor and the foreach path), a mid-run state_dict hand-over in both directions, and the folded gradient scale."""
    import rnd_semantic_segmentation_b200 as b200
    g = torch.Generator().manual_seed(8)
    shapes = [(19, 256, 3, 3), (19,)] * 4 + [(33, 5)] * 12
    p0 = [torch.randn(s, generator=g).cuda() * 0.05 for s in shapes]
    grads = [[torch.randn(s, generator=g).cuda() * 0.01 for s in shapes] for _ in range(5)]
    fused_cls = b200.FusedSGD if kind == "sgd" else b200.FusedAdam
    torch_cls = torch.optim.SGD if kind == "sgd" else torch.optim.Adam

    def steps(opt, ps, ks, scale=1.0):
        for k in ks:
            for p, gr in zip(ps, grads[k]):
                p.grad = gr.clone() * scale
            opt.step()

    def fresh():
        return [torch.nn.Parameter(p.clone()) for p in p0]

    pa, pb, pc = fresh(), fresh(), fresh()
    oa, ob, oc = fused_cls(pa, **hyper), torch_cls(pb, foreach=False, **hyper), torch_cls(pc, foreach=True, **hyper)
    steps(oa, pa, range(5)); steps(ob, pb, range(5)); steps(oc, pc, range(5))
    for a, b, c in zip(pa, pb, pc):
        assert rel_err(a, b) <= OPT_TOL and rel_err(a, c) <= OPT_TOL
    # hand-over: 2 steps torch -> state_dict -> 3 steps fused, and the other way round
    pd_, pe = fresh(), fresh()
    od, oe = torch_cls(pd_, foreach=False, **hyper), fused_cls(pe, **hyper)
    steps(od, pd_, range(2))
    with torch.no_grad():
        for e, d in zip(pe, pd_):
            e.copy_(d)
    oe.load_state_dict(od.state_dict())
    steps(oe, pe, range(2, 5))
    for e, b in zip(pe, pb):
        assert rel_err(e, b) <= OPT_TOL
    pf, pg = fresh(), fresh()
    of, og = fused_cls(pf, **hyper), torch_cls(pg, foreach=False, **hyper)
    steps(of, pf, range(2))
    with torch.no_grad():
        for t, f in zip(pg, pf):
            t.copy_(f)
    og.load_state_dict(of.state_dict())
    steps(og, pg, range(2, 5))
    for t, b in zip(pg, pb):
        assert rel_err(t, b) <= OPT_TOL
    # gradient scale folded into the step == scaling the gradients first (DDP mean after a SUM all-reduce over 8 ranks)
    ph = fresh()
    oh = fused_cls(ph, grad_scale=0.125, **hyper)
    steps(oh, ph, range(5), scale=8.0)
    for h_, a in zip(ph, pa):
        assert rel_err(h_, a) <= OPT_TOL


def test_k8_rejects_cpu_parameters(lib):
    import rnd_semantic_segmentation_b200 as b200
    p = torch.nn.Parameter(torch.zeros(4))
    p.grad = torch.ones(4)
    for cls, kw in ((b200.FusedSGD, dict(lr=0.1, momentum=0.9)), (b200.FusedAdam, dict(lr=0.1))):
        with pytest.raises(lib.B200SegError):
            cls([p], **kw).step()


def test_k8_step_invalidates_packed_weight_caches(lib):
    """The kernels update parameters through raw pointers; the modules cache their packed bf16 weights keyed on the parameters'
    version counters, so a fused step must bump them: the next forward uses the updated weights."""
    import rnd_semantic_segmentation_b200 as b200
    torch.manual_seed(12)
    head = b200.ASPP_Classifier_V2(64, RATES, RATES, 19).cuda()
    D = b200.PixelDiscriminator(64, 16, num_classes=19).cuda()
    x = torch.relu(torch.randn(1, 64, 20, 24, device="cuda"))
    for mod, opt in ((head, b200.FusedSGD(head.parameters(), lr=0.5, momentum=0.9)), (D, b200.FusedAdam(D.parameters(), lr=0.05))):
        for step in range(2):                                 # first step (state creation path) and a planned step
            with torch.no_grad():
                before = mod(x).clone()
            versions = [p._version for p in mod.parameters()]
            for p in mod.parameters():
                p.grad = torch.randn_like(p)
            opt.step()
            assert all(p._version > v for p, v in zip(mod.parameters(), versions))
            with torch.no_grad():
                after = mod(x)
            fresh = type(mod)(64, RATES, RATES, 19) if mod is head else type(mod)(64, 16, num_classes=19)
            fresh.load_state_dict(mod.state_dict())
            fresh.cuda()
            with torch.no_grad():
                want = fresh(x)
            assert not torch.equal(after, before) and torch.equal(after, want), (type(mod).__name__, step)


def test_k8_unaligned_views_and_two_launch_groups(lib):
    """25 parameters that are 4-byte-aligned views into one buffer (scalar head/tail paths, > 16 tensors = two launches, lengths
    1 .. 4097) with guard elements between them: the update equals torch.optim's and nothing outside the views is touched."""
    import rnd_semantic_segmentation_b200 as b200
    g = torch.Generator().manual_seed(21)
    shapes = [(19, 64, 3, 3), (19,), (4097,), (3, 5), (1,)] * 5
    total = sum(torch.Size(s).numel() + 3 for s in shapes) + 8
    for kind, hyper in (("sgd", dict(lr=0.1, momentum=0.9, weight_decay=1e-3)), ("adam", dict(lr=1e-3, betas=(0.9, 0.99)))):
        base0 = torch.randn(total, generator=g)
        base = base0.clone().cuda()
        ours, refs, mask, off = [], [], torch.zeros(total, dtype=torch.bool), 1
        for s in shapes:
            nel = torch.Size(s).numel()
            ours.append(torch.nn.Parameter(base[off:off + nel].view(s)))
            refs.append(torch.nn.Parameter(base0[off:off + nel].view(s).clone().cuda()))
            mask[off:off + nel] = True
            off += nel + 3                                   # three guard elements after every tensor
        oa = (b200.FusedSGD if kind == "sgd" else b200.FusedAdam)(ours, **hyper)
        ob = (torch.optim.SGD if kind == "sgd" else torch.optim.Adam)(refs, foreach=False, **hyper)
        for _ in range(3):
            for a, b in zip(ours, refs):
                gr = torch.randn(a.shape, generator=g).cuda()
                a.grad, b.grad = gr.clone(), gr.clone()
            oa.step(); ob.step()
        for a, b in zip(ours, refs):
            assert rel_err(a, b) <= OPT_TOL
        assert torch.equal(base.cpu()[~mask], base0[~mask])     # guards untouched


@pytest.mark.parametrize("C,shapes,flips,divisors,H,W", [
    (19, [(64, 128), (64, 128)], [False, True], (2,), 512, 1024),
    (19, [(33, 65), (17, 40)], [True, False], (2,), 263, 517),            # members of different sizes, ragged strip and row block
    (2, [(44, 44)], [True], (), 352, 352),
    (7, [(9, 11), (9, 11)], [False, True], (2,), 5, 300),                 # fewer rows than a row block
    (30, [(8, 8), (12, 10)], [False, False], (2,), 64, 61),
    (19, [(8, 8)], [False], (), 8, 8),                                    # no upsampling at all: every row changes the source pair
    (19, [(23, 45), (33, 65), (43, 84)], [False, True, False], (3,), 260, 517),       # three and four members (multi-scale)
    (5, [(9, 9), (12, 14), (12, 14), (20, 17)], [False, False, True, True], (2, 2), 77, 130),
])
def test_k7_row_walking_kernel_equals_per_pixel_kernel(lib, C, shapes, flips, divisors, H, W):
    """Ensembles of <= 4 members run the row-walking kernel (source-row lerps cached per thread in shared memory); the per-pixel
    kernel (larger ensembles) must give bit-identical probabilities, labels and counts, and both must equal torch."""
    members = _tta_members(C, shapes, 1.0, seed=400 + C + H)
    labels = make_labels(1, H, W, C, 0.1, 23).cuda()
    outs = []
    for row_walk in (True, False):
        lib.tta_set_row_walk(row_walk)
        try:
            outs.append(lib.tta_argmax_confusion(members, flips, (H, W), labels=labels, divisors=divisors, want_pred=True, want_probs=True))
        finally:
            lib.tta_set_row_walk(True)
    (cm_a, pred_a, probs_a), (cm_b, pred_b, probs_b) = outs
    assert torch.equal(probs_a, probs_b) and torch.equal(pred_a, pred_b) and torch.equal(cm_a, cm_b)
    assert torch.equal(probs_a.unsqueeze(0), to.tta_probabilities(members, flips, (H, W), divisors))


def test_pseudo_label_map_and_png_writer(lib, tmp_path):
    """save_distill's argmax (aspp_tester.py:40-42) through the fused kernels: equal to the argmax of the materialised
    probabilities for a plain frame (K4) and for the flip ensemble (K7); the PNG holds exactly those labels."""
    import rnd_semantic_segmentation_b200 as b200
    from PIL import Image
    g = torch.Generator().manual_seed(31)
    label = torch.zeros(1, 120, 200, dtype=torch.int64).cuda()
    both = torch.randn(2, 19, 15, 25, generator=g).cuda()
    palette = list(range(256)) * 3
    outs = {
        "plain": b200.utility.LazyProbabilities(both[:1].contiguous(), label),
        "flip": b200.utility.LazyProbabilities(None, label, members=[both[0:1].contiguous(), both[1:2].contiguous()], flips=[False, True],
                                               divisors=(2,)),
    }
    for name, out in outs.items():
        want = out.materialize().cpu().numpy().squeeze().argmax(0)           # the reference's save_distill arithmetic
        got = b200.pseudo_label_map(out)
        assert got.dtype == np.uint8 and got.shape == (120, 200)
        np.testing.assert_array_equal(got, want.astype(np.uint8))
        path = tmp_path / f"{name}.png"
        b200.save_pseudo_label(out, str(path), palette)
        np.testing.assert_array_equal(np.asarray(Image.open(path)), got)


@pytest.mark.parametrize("C,Cin,R", [(19, 2048, 4), (2, 64, 4), (30, 128, 3), (7, 24, 1)])
def test_head_weight_pack_layouts_exact(lib, C, Cin, R):
    """Wp [NJ,Cin] / WpT [Cin,NJ] / bias_sum of the tiled pack kernel against the layout definition built with torch: rows
    (r*8+q)*C + c = the 8 off-centre taps of branch r, rows 8R*C + c = the fp32 sum of the R centre taps, rounded once to bf16;
    padding rows zero."""
    g = torch.Generator().manual_seed(C + Cin)
    ws = [(torch.randn(C, Cin, 3, 3, generator=g) * 0.05).cuda() for _ in range(R)]
    bs = [torch.randn(C, generator=g).cuda() for _ in range(R)]
    Wp, WpT, bias_sum = lib.aspp_pack_weights(ws, bs)
    NJ = Wp.shape[0]
    want = torch.zeros(NJ, Cin, device="cuda")
    for r in range(R):
        flat = ws[r].reshape(C, Cin, 9)
        for q in range(8):
            k = q if q < 4 else q + 1
            want[(r * 8 + q) * C:(r * 8 + q + 1) * C] = flat[:, :, k]
    centre = ws[0].reshape(C, Cin, 9)[:, :, 4].clone()
    for r in range(1, R):
        centre = centre + ws[r].reshape(C, Cin, 9)[:, :, 4]
    want[8 * R * C:(8 * R + 1) * C] = centre
    want = want.to(torch.bfloat16)
    assert torch.equal(Wp, want) and torch.equal(WpT, want.t().contiguous())
    bsum = bs[0].clone()
    for r in range(1, R):
        bsum = bsum + bs[r]
    assert torch.equal(bias_sum, bsum)


@pytest.mark.parametrize("parts,Ci", [([256], 2048), ([19, 19], 128), ([40], 64), ([16], 24), ([5, 3], 72)])
def test_conv_weight_pack_layouts_exact(lib, parts, Ci):
    g = torch.Generator().manual_seed(sum(parts) + Ci)
    ws = [(torch.randn(co, Ci, 3, 3, generator=g) * 0.05).cuda() for co in parts]
    Wf, Wb = lib.conv3x3_pack_weights(ws)
    allw = torch.cat(ws, 0).reshape(sum(parts), Ci, 9).to(torch.bfloat16)          # [Co, Ci, 9]
    assert torch.equal(Wf, allw.permute(2, 0, 1).contiguous())
    Co = sum(parts)
    assert torch.equal(Wb[:, :, :Co], allw.permute(2, 1, 0).contiguous()) and float(Wb[:, :, Co:].abs().sum()) == 0.0


@pytest.mark.parametrize("C,shapes,flips,divisors,H,W,sigma", [
    (19, [(64, 128), (64, 128)], [False, True], (2,), 512, 1024, 1.0),
    (19, [(64, 128), (64, 128)], [False, True], (2,), 512, 1024, 0.01),       # near-uniform probabilities: many near ties
    (19, [(23, 45), (33, 65), (43, 84)], [False, True, False], (3,), 260, 517, 0.01),
    (2, [(44, 44), (44, 44)], [False, True], (2,), 352, 352, 0.01),
    (7, [(9, 11)], [True], (), 50, 70, 1e-4),
    (20, [(8, 8), (12, 10)], [False, False], (2,), 64, 61, 0.01),
])
def test_k7_labels_only_fast_path_is_bit_exact(lib, C, shapes, flips, divisors, H, W, sigma):
    """Without a probability output the row-walking kernel orders the classes with ex2.approx-based probabilities and re-runs the
    exact sequence only on near ties: labels and confusion matrix must equal the exact kernel's and torch's, bit for bit."""
    members = _tta_members(C, shapes, sigma, seed=500 + C + len(shapes))
    labels = make_labels(1, H, W, C, 0.1, 29).cuda()
    want_pred = to.tta_probabilities(members, flips, (H, W), divisors).max(1)[1]
    got = {}
    for fast in (True, False):
        lib.tta_set_row_walk(True, fast=fast)
        try:
            got[fast] = lib.tta_argmax_confusion(members, flips, (H, W), labels=labels, divisors=divisors, want_pred=True)
        finally:
            lib.tta_set_row_walk(True)
    assert torch.equal(got[True][1], got[False][1]) and torch.equal(got[True][0], got[False][0])
    assert torch.equal(got[True][1].unsqueeze(0), want_pred)
    cm_only, _, _ = lib.tta_argmax_confusion(members, flips, (H, W), labels=labels, divisors=divisors)
    assert torch.equal(cm_only.cpu(), to.confusion_matrix_bincount(C, want_pred.flatten().cpu(), labels.flatten().cpu()))


def test_k7_fast_path_exact_ties_and_one_ulp_pairs(lib):
    """Adversarial members: identical classes (exact ties -> first index), pairs one ulp apart, and a member whose mirror image
    cancels the other's preference -- the fast path has to hand every such pixel to the exact sequence."""
    torch.manual_seed(5)
    base = torch.randn(1, 1, 16, 32).repeat(1, 19, 1, 1)
    base[:, 5] = torch.nextafter(base[:, 5], torch.full_like(base[:, 5], 10.0))
    base[:, 11] = base[:, 5]
    a = base.cuda()
    b = base.flip(3).contiguous().cuda()                      # mirrored twin: un-mirrored it equals a (up to sampling rounding)
    labels = make_labels(1, 128, 256, 19, 0.2, 9).cuda()
    for members, flips, divs in (([a], [False], ()), ([a, b], [False, True], (2,)), ([a, a], [False, False], (2,))):
        want = to.tta_probabilities(members, flips, (128, 256), divs).max(1)[1]
        cm, pred, _ = lib.tta_argmax_confusion(members, flips, (128, 256), labels=labels, divisors=divs, want_pred=True)
        assert torch.equal(pred.unsqueeze(0), want)
        assert torch.equal(cm.cpu(), to.confusion_matrix_bincount(19, want.flatten().cpu(), labels.flatten().cpu()))
