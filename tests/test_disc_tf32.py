"""TF32 PixelDiscriminator (``PixelDiscriminator.tf32``): the conv stack's tcgen05 implicit GEMMs with kind::tf32 operands and fp32
activations / gradients.  CPU: the flag's plumbing (default, state_dict, deepcopy / save-load, install(disc_tf32=True)).  GPU: every
layer against an fp64 convolution of the TF32-rounded operands, the whole stack against the fp64 reference module next to torch's own
cuDNN TF32 stack, and the FADA iterations with optimizer steps against the oracle."""
import copy
import inspect
import sys
import types

import pytest
import torch
import torch.nn.functional as F

import rnd_semantic_segmentation_b200 as b200
from helpers import RATES, make_labels, rel_err
from oracle import torch_oracle as to


def tf32_round(t):
    """fp32 -> nearest TF32 value, ties to even (low 13 mantissa bits cleared), as the kernels store it."""
    u = t.float().contiguous().view(torch.int32)
    r = (u + 0xFFF + ((u >> 13) & 1)) & -8192
    finite = torch.isfinite(t.float())
    return torch.where(finite, r, u).view(torch.float32)


def low_bits_zero(t):
    return int((t.detach().float().contiguous().view(torch.int32) & 0x1FFF).abs().max()) == 0


# ------------------------------------------------------------------ CPU: the flag
def test_flag_default_state_dict_deepcopy_and_save_load(tmp_path):
    D = b200.PixelDiscriminator(64, 32, num_classes=3)
    assert D.tf32 is False
    keys = set(D.state_dict().keys())
    D.tf32 = True
    assert set(D.state_dict().keys()) == keys and not any("tf32" in k for k in keys)
    assert copy.deepcopy(D).tf32 is True
    path = tmp_path / "d.pt"
    torch.save(D, path)
    assert torch.load(path, weights_only=False).tf32 is True
    plain = b200.PixelDiscriminator(64, 32, num_classes=3)
    plain.load_state_dict(D.state_dict())                        # checkpoints interchange across precisions
    assert plain.tf32 is False
    old = b200.PixelDiscriminator.__new__(b200.PixelDiscriminator)   # a module pickled before the flag existed
    assert old.tf32 is False


def test_install_disc_tf32_wraps_the_factory(monkeypatch):
    core = types.ModuleType("core"); models = types.ModuleType("core.models"); bld = types.ModuleType("core.models.build")
    for m in (core, models, bld):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    cfg = types.SimpleNamespace(MODEL=types.SimpleNamespace(NAME="deeplab_resnet101", NUM_CLASSES=3))
    b200.install()
    assert bld.build_adversarial_discriminator is b200.build_adversarial_discriminator
    assert bld.build_adversarial_discriminator(cfg, 64, 32).tf32 is False
    b200.install(disc_tf32=True)
    fn = bld.build_adversarial_discriminator
    assert fn is not b200.build_adversarial_discriminator and models.build_adversarial_discriminator is fn
    assert inspect.signature(fn) == inspect.signature(b200.build_adversarial_discriminator)
    D = fn(cfg, 64, 32)
    assert isinstance(D, b200.PixelDiscriminator) and D.tf32 is True
    b200.install(disc_tf32=True)
    assert bld.build_adversarial_discriminator is fn                  # the same wrapper, not wrapped twice
    b200.install()
    assert bld.build_adversarial_discriminator(cfg, 64, 32).tf32 is False


def test_abi_table_lists_the_tf32_entries():
    from rnd_semantic_segmentation_b200 import _lib
    for name in ("b200seg_disc_forward_tf32", "b200seg_disc_backward_tf32", "b200seg_disc_backward_tf32_scratch_bytes",
                 "b200seg_conv3x3_forward_tf32", "b200seg_conv3x3_dgrad_tf32", "b200seg_conv3x3_wgrad_tf32",
                 "b200seg_conv3x3_pack_weights_stack_tf32"):
        assert name in _lib.SIGNATURES


def test_tf32_round_helper():
    x = torch.tensor([1.0, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, -(1.0 + 2.0 ** -11), float("inf"), 0.0])
    want = torch.tensor([1.0, 1.0, 1.0 + 4 * 2.0 ** -11, -1.0, float("inf"), 0.0])         # ties to even
    assert torch.equal(tf32_round(x), want)


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lib():
    from rnd_semantic_segmentation_b200 import _lib
    _lib.load()
    return _lib


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous().float().cuda()


def _nchw(t):
    return t.float().cpu().permute(0, 3, 1, 2)


def _pack(lib, wt):
    (pair,), _ = lib.conv3x3_pack_weights_stack([[wt.cuda()]], tf32=True)
    return pair


@pytest.mark.gpu
@pytest.mark.parametrize("n,ci,co,h,w,dil", [
    (2, 128, 256, 64, 128, 1), (1, 256, 128, 33, 65, 1), (2, 64, 40, 9, 11, 1), (1, 24, 16, 20, 27, 1), (1, 192, 64, 17, 40, 2),
    (4, 2048, 256, 64, 128, 1),      # the adversarial layer at full size
])
def test_tf32_conv3x3_layer(lib, n, ci, co, h, w, dil):
    full = ci == 2048
    g = torch.Generator().manual_seed(300 + h + ci)
    x = tf32_round(torch.randn(n, ci, h, w, generator=g))
    wt = torch.randn(co, ci, 3, 3, generator=g) * (0.01 if full else 0.05)
    b = torch.randn(co, generator=g) * 0.1
    go = tf32_round(torch.randn(n, co, h, w, generator=g))
    mask_src = tf32_round(torch.randn(n, ci, h, w, generator=g))
    mask_src[0, 0, 0, :3] = 0.0                                     # LeakyReLU'(0) = slope
    Wf, Wb = _pack(lib, wt)
    wq = tf32_round(wt)
    assert torch.equal(Wf.cpu(), wq.permute(2, 3, 0, 1).reshape(9, co, ci))
    # fp64 reference on the device (the full-size layer is 1.2 TFLOP a direction)
    xd, wd = x.double().cuda().requires_grad_(True), wq.double().cuda().requires_grad_(True)
    z = F.conv2d(xd, wd, b.double().cuda(), padding=dil, dilation=dil)
    gx_want, gw_want = torch.autograd.grad(z, (xd, wd), go.double().cuda())
    z = z.detach()
    xq, gq, mq = _nhwc(x), _nhwc(go), _nhwc(mask_src)
    mfac = torch.where(mask_src > 0, 1.0, 0.2).double().cuda()
    runs = {}
    for pair in (True, False):
        lib.conv_set_pair(pair)
        try:
            r = {}
            r["fwd_nchw"] = lib.conv3x3_forward(xq, Wf, b.cuda(), None, dilation=dil, out_f32_nchw=True)
            r["fwd_nhwc"] = lib.conv3x3_forward(xq, Wf, b.cuda(), 0.2, dilation=dil)
            r["dgrad_nchw"] = lib.conv3x3_dgrad(gq, Wb, dilation=dil, out_f32_nchw=True)
            r["dgrad_nhwc"], r["colsum"] = lib.conv3x3_dgrad(gq, Wb, mask=mq, slope=0.2, dilation=dil, want_colsum=True)
            r["dgrad_nhwc_plain"] = lib.conv3x3_dgrad(gq, Wb, mask=mq, slope=0.2, dilation=dil)
            for splits in (0, 1, 3):
                r[f"wgrad{splits}"], = lib.conv3x3_wgrad(gq, xq, [co], dilation=dil, splits=splits)
            again = lib.conv3x3_forward(xq, Wf, b.cuda(), 0.2, dilation=dil)
            assert torch.equal(again, r["fwd_nhwc"])                            # run to run
            assert torch.equal(lib.conv3x3_wgrad(gq, xq, [co], dilation=dil)[0], r["wgrad0"])
        finally:
            lib.conv_set_pair(True)
        runs[pair] = r
        errs = {"fwd_nchw": rel_err(r["fwd_nchw"], z), "dgrad_nchw": rel_err(r["dgrad_nchw"], gx_want)}
        for splits in (0, 1, 3):
            errs[f"wgrad{splits}"] = rel_err(r[f"wgrad{splits}"], gw_want)
        errs["fwd_nhwc"] = rel_err(_nchw(r["fwd_nhwc"]), F.leaky_relu(z, 0.2))
        errs["dgrad_nhwc"] = rel_err(_nchw(r["dgrad_nhwc"]), gx_want * mfac)
        errs["colsum"] = rel_err(r["colsum"], (gx_want * mfac).sum((0, 2, 3)))
        print(f"pair={pair}", {k: f"{v:.2e}" for k, v in errs.items()})
        # 2e-5 per 4096 terms of one fp32 accumulation in TMEM: the full-size forward sums K = 18 432 and a single-split weight
        # gradient sums every pixel (measured up to 4.8e-5 at K = 16 384)
        k_len = {"fwd_nchw": 9 * ci, "dgrad_nchw": 9 * co, "wgrad0": n * h * w, "wgrad1": n * h * w, "wgrad3": -(-n * h * w // 3)}
        for k in ("fwd_nchw", "dgrad_nchw", "wgrad0", "wgrad1", "wgrad3"):
            assert errs[k] <= 2e-5 * max(1.0, k_len[k] / 4096), (pair, k, errs[k])
        assert errs["fwd_nhwc"] <= 5e-4 and errs["dgrad_nhwc"] <= 5e-4, (pair, errs)
        assert errs["colsum"] <= 1e-5, (pair, errs)
        assert low_bits_zero(r["fwd_nhwc"]) and low_bits_zero(r["dgrad_nhwc"])
        assert torch.equal(r["dgrad_nhwc"], r["dgrad_nhwc_plain"])
        # the stored tensors are the rounding of the unrounded results
        assert torch.equal(r["fwd_nhwc"], tf32_round(F.leaky_relu(r["fwd_nchw"], 0.2)).permute(0, 2, 3, 1).contiguous())
    for k in runs[True]:
        assert torch.equal(runs[True][k], runs[False][k]), k                    # pair and single-CTA modes: the same bits


def _stack_reference(ref64, x, go, slope=0.2):
    xr = x.double().requires_grad_(True)
    out = ref64(xr)
    out.backward(go.double())
    return out.detach(), xr.grad, [p.grad.clone() for p in ref64.parameters()]


@pytest.mark.gpu
@pytest.mark.parametrize("n,cin,ndf,C,h,w", [(2, 256, 64, 19, 33, 65), (1, 2048, 256, 19, 32, 64), (2, 64, 32, 2, 44, 44), (1, 24, 16, 3, 20, 27)])
def test_tf32_stack_against_fp64_and_cudnn_tf32(lib, n, cin, ndf, C, h, w):
    torch.manual_seed(40 + C)
    ref = to.PixelDiscriminatorOracle(cin, ndf, num_classes=C)
    ours = b200.PixelDiscriminator(cin, ndf, num_classes=C)
    ours.load_state_dict(ref.state_dict())
    ours.tf32 = True
    ours.cuda()
    g = torch.Generator().manual_seed(41 + h)
    x = torch.relu(torch.randn(n, cin, h, w, generator=g))
    go = torch.randn(n, 2 * C, h, w, generator=g) * 1e-3
    want_out, want_gx, want_gp = _stack_reference(copy.deepcopy(ref).double(), x, go)
    # torch's own stack on the GPU under allow_tf32 (what the reference runs), on the same inputs
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True
    try:
        cud = copy.deepcopy(ref).cuda()
        xc_ref = x.cuda().requires_grad_(True)
        out_c = cud(xc_ref)
        out_c.backward(go.cuda())
    finally:
        torch.backends.cudnn.allow_tf32 = old
    xc = x.cuda().requires_grad_(True)
    got = ours(xc)
    got.backward(go.cuda())
    # LeakyReLU sign disagreements between the stored TF32 activations and an fp64 chain of the same roundings
    with torch.no_grad():
        (Wf1, _), (Wf2, _), _, _ = ours._packed_weights()
        A1 = lib.conv3x3_forward(_nhwc(tf32_round(x)), Wf1, ours.D[0].bias.detach(), 0.2)
        A2 = lib.conv3x3_forward(A1, Wf2, ours.D[2].bias.detach(), 0.2)
        r = lambda t: tf32_round(t.float()).double()  # noqa: E731
        z1 = F.conv2d(r(x), r(ref.D[0].weight.detach()), ref.D[0].bias.detach().double(), padding=1)
        z2 = F.conv2d(r(F.leaky_relu(z1, 0.2)), r(ref.D[2].weight.detach()), ref.D[2].bias.detach().double(), padding=1)
        flips = int(((_nchw(A1) > 0) != (z1 > 0)).sum()) + int(((_nchw(A2) > 0) != (z2 > 0)).sum())
        n_act = z1.numel() + z2.numel()
    print(f"LeakyReLU sign disagreements: {flips} of {n_act}")
    assert flips <= max(2, int(1e-4 * n_act)), (flips, n_act)
    pairs = [("logits", got, out_c, want_out), ("x.grad", xc.grad, xc_ref.grad, want_gx)]
    pairs += [(name, p.grad, pc.grad, pw) for (name, p), pc, pw in zip(ours.named_parameters(), cud.parameters(), want_gp)]
    for name, a, c, wnt in pairs:
        e_ours, e_cudnn = rel_err(a, wnt), rel_err(c, wnt)
        print(f"{name:12s} TF32 K6 {e_ours:.2e}   cuDNN allow_tf32 {e_cudnn:.2e}")
        assert e_ours <= max(2 * e_cudnn, 2e-3), (name, e_ours, e_cudnn)


@pytest.mark.gpu
def test_tf32_seam_input_eval_toggle_and_default_unchanged(lib):
    torch.manual_seed(5)
    n, cin, ndf, C, h, w = 2, 256, 64, 19, 33, 65
    D = b200.PixelDiscriminator(cin, ndf, num_classes=C).cuda()
    g = torch.Generator(device="cuda").manual_seed(6)
    x_bf = torch.relu(torch.randn(n, cin, h, w, device="cuda", generator=g)).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    x_f = x_bf.float().contiguous()
    go = torch.randn(n, 2 * C, h, w, device="cuda", generator=g) * 1e-3
    # without the flag: bit-identical to a direct call of the bf16 one-call entry
    out_default = D(x_f)
    out_direct = lib.disc_forward(x_f, 0, (n, cin, h, w), (D.D[0].weight, D.D[2].weight, D.cls1.weight, D.cls2.weight),
                                  (D.D[0].bias, D.D[2].bias, D.cls1.bias, D.cls2.bias), 0.2)[0]
    assert torch.equal(out_default, out_direct)
    # bf16 channels_last features equal fp32 NCHW features holding the same values; x.grad keeps the input's format
    D.tf32 = True
    xa, xb = x_bf.clone().requires_grad_(True), x_f.clone().requires_grad_(True)
    oa, ob = D(xa), D(xb)
    assert torch.equal(oa, ob)
    ga = torch.autograd.grad(oa, (xa, *D.parameters()), go)
    gb = torch.autograd.grad(ob, (xb, *D.parameters()), go)
    assert ga[0].dtype == torch.bfloat16 and ga[0].is_contiguous(memory_format=torch.channels_last)
    assert gb[0].dtype == torch.float32 and gb[0].is_contiguous()
    assert torch.equal(ga[0], gb[0].to(torch.bfloat16))
    assert all(torch.equal(a, b) for a, b in zip(ga[1:], gb[1:]))
    # eval mode: flipping the flag never reuses the other precision's cached pack
    D.eval()
    with torch.no_grad():
        e_tf = D.logits(x_f)
        D.tf32 = False
        e_bf = D.logits(x_f)
        D.tf32 = True
        e_tf2 = D.logits(x_f)
    assert torch.equal(e_tf, ob.detach()) and torch.equal(e_bf, out_default) and torch.equal(e_tf2, e_tf)
    assert not torch.equal(e_tf, e_bf)


@pytest.mark.gpu
def test_tf32_loss_step_cuda_graph_replay(lib):
    torch.manual_seed(8)
    n, cin, ndf, C, h, w, H, W = 2, 256, 64, 19, 16, 32, 128, 256
    D = b200.PixelDiscriminator(cin, ndf, num_classes=C).cuda()
    D.tf32 = True
    D_eager = copy.deepcopy(D)
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.relu(torch.randn(n, cin, h, w, device="cuda", generator=g))
    seg = torch.randn(n, C, h, w, device="cuda", generator=g)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            D.zero_grad(set_to_none=True)
            D.forward_soft_loss(x, seg, (H, W), slot=1).backward()
    torch.cuda.current_stream().wait_stream(s)
    D.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = D.forward_soft_loss(x, seg, (H, W), slot=1)
        loss.backward()
    x.copy_(torch.relu(torch.randn(n, cin, h, w, device="cuda", generator=g)))
    seg.copy_(torch.randn(n, C, h, w, device="cuda", generator=g))
    graph.replay()
    torch.cuda.synchronize()
    want = D_eager.forward_soft_loss(x, seg, (H, W), slot=1)
    want.backward()
    assert torch.equal(loss, want)
    assert all(torch.equal(p.grad, q.grad) for p, q in zip(D.parameters(), D_eager.parameters()))


@pytest.mark.gpu
def test_tf32_fada_iterations_with_optimizer_steps_match_oracle(lib):
    """test_fada_iterations_with_optimizer_steps_match_oracle with D.tf32 = True: losses within 5e-3, discriminator gradients of the
    first iteration within 1e-2 in L2 (bf16: 3e-2; later iterations start from parameters the two Adam runs have already moved
    apart), and updates after three iterations within the bf16 bar of 0.1 in L2.  The updates do not tighten with the gradients:
    Adam's first steps are lr * m / sqrt(v), close to lr * sign(g), so an element whose gradient is near zero moves by a full step
    either way and the L2 difference counts those sign decisions (measured on a B200: 9.8e-2 for D.0.bias, 256 elements;
    4.8e-2 for D.0.weight)."""
    n, cin, C, h, w, H, W = 2, 256, 19, 16, 32, 128, 256
    torch.manual_seed(91)
    ref_head = to.AsppHeadOracle(cin, RATES, RATES, C)
    ref_D = to.PixelDiscriminatorOracle(cin, 64, num_classes=C)
    head = b200.ASPP_Classifier_V2(cin, RATES, RATES, C)
    head.load_state_dict(ref_head.state_dict())
    D = b200.PixelDiscriminator(cin, 64, num_classes=C)
    D.load_state_dict(ref_D.state_dict())
    D.tf32 = True
    head.cuda(), D.cuda()
    D0 = copy.deepcopy(ref_D.state_dict())
    base_lr, base_lr_d, max_iter = 2.5e-4, 1e-4, 10
    ref_cls = torch.optim.SGD(ref_head.parameters(), lr=base_lr * 10, momentum=0.9, weight_decay=5e-4)
    ref_opt_d = torch.optim.Adam(ref_D.parameters(), lr=base_lr_d, betas=(0.9, 0.99))
    opt_cls = b200.FusedSGD(head.parameters(), lr=base_lr * 10, momentum=0.9, weight_decay=5e-4)
    opt_d = b200.FusedAdam(D.parameters(), lr=base_lr_d, betas=(0.9, 0.99))
    g = torch.Generator().manual_seed(92)
    size = (H, W)
    worst_loss, worst_grad = 0.0, 0.0
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
            e = abs(got.item() - exp.item()) / abs(exp.item())
            worst_loss = max(worst_loss, e)
            assert e <= 5e-3, (it, name, got.item(), exp.item())
        for (name, p), pr in zip(D.named_parameters(), ref_D.parameters()):
            got, exp = p.grad.detach().cpu().double(), pr.grad.double()
            e = ((got - exp).norm() / exp.norm()).item()
            print(f"iteration {it} {name} gradient L2 {e:.2e}")
            if it == 0:
                worst_grad = max(worst_grad, e)
                assert e <= 1e-2, (it, name, e)
    upd = {}
    for (name, p), pr in zip(D.named_parameters(), ref_D.parameters()):
        d_got, d_exp = p.detach().cpu().double() - D0[name].double(), pr.detach().double() - D0[name].double()
        assert float(d_exp.norm()) > 0, name
        upd[name] = ((d_got - d_exp).norm() / d_exp.norm()).item()
    print("D-update L2 after three iterations:", {k: f"{v:.2e}" for k, v in upd.items()})
    worst_upd = max(upd.values())
    assert worst_upd <= 0.1, upd
    print(f"TF32 FADA: worst loss rel {worst_loss:.2e}, worst first-iteration D-gradient L2 {worst_grad:.2e}, "
          f"worst D-update L2 {worst_upd:.2e}")
