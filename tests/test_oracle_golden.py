"""The oracle (oracle/torch_oracle.py, oracle/np_oracle.py) against the golden vectors
generated from the reference's own code (oracle/gen_golden.py) -- CPU only."""
import numpy as np
import pytest
import torch

from oracle import np_oracle as npo
from oracle import torch_oracle as to

RATES = [6, 12, 18, 24]


def _head_from_golden(g, cin, ncls):
    head = to.AsppHeadOracle(cin, RATES, RATES, ncls)
    sd = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")}
    assert list(sd.keys()) == list(head.state_dict().keys())       # key names + order = checkpoint contract
    head.load_state_dict(sd)
    return head


@pytest.mark.parametrize("name", ["head_c19", "head_c2", "head_c19_T18"])
def test_head_ce_matches_reference_golden(golden, name):
    g = golden(name)
    x = torch.from_numpy(g["x"])
    labels = torch.from_numpy(g["labels"])
    ncls = int(g["num_classes"])
    head = _head_from_golden(g, x.shape[1], ncls)
    with torch.no_grad():
        np.testing.assert_allclose(head(x).numpy(), g["logits_lr"], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(head(x, labels.shape[-2:]).numpy(), g["logits_hr"], rtol=1e-5, atol=1e-6)
    loss, gx, gparams = to.train_step_src(head, x, labels, temperature=float(g["temperature"]))
    assert abs(loss.item() - float(g["loss"])) <= 1e-6 * max(1.0, abs(float(g["loss"])))
    np.testing.assert_allclose(gx.numpy(), g["grad_x"], rtol=1e-4, atol=1e-8)
    for (k, _), gp in zip(head.named_parameters(), gparams):
        np.testing.assert_allclose(gp.numpy(), g["grad." + k], rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("name", ["head_c19", "head_c2"])
def test_numpy_restatement_matches_golden(golden, name):
    g = golden(name)
    ws = [g[f"sd.conv2d_list.{i}.weight"] for i in range(4)]
    bs = [g[f"sd.conv2d_list.{i}.bias"] for i in range(4)]
    lr = npo.aspp_head(g["x"], ws, bs)
    np.testing.assert_allclose(lr, g["logits_lr"], rtol=1e-4, atol=1e-5)
    hr = npo.upsample_bilinear_ac(g["logits_lr"], g["labels"].shape[-2:])
    np.testing.assert_allclose(hr, g["logits_hr"], rtol=1e-5, atol=2e-6)
    loss, n_valid = npo.hard_cross_entropy(g["logits_hr"] / float(g["temperature"]), g["labels"])
    assert abs(loss - float(g["loss"])) < 2e-6
    # gradient chain: CE grad -> bilinear adjoint == d loss / d low-res logits; check through the
    # bias gradient (sum over pixels of the low-res grad) which the golden holds per conv.
    g_hr = npo.hard_cross_entropy_grad(g["logits_hr"] / float(g["temperature"]), g["labels"]) / float(g["temperature"])
    g_lr = npo.upsample_bilinear_ac_adjoint(g_hr, g["logits_lr"].shape[-2:])
    np.testing.assert_allclose(g_lr.sum(axis=(0, 2, 3)), g["grad.conv2d_list.0.bias"], rtol=2e-4, atol=1e-7)


def test_all_ignored_is_nan(golden):
    g = golden("head_all_ignored")
    assert np.isnan(g["loss"])
    head = _head_from_golden(g, g["x"].shape[1], int(g["num_classes"]))
    loss = to.hard_cross_entropy(head(torch.from_numpy(g["x"]), (20, 20)), torch.from_numpy(g["labels"]))
    assert torch.isnan(loss)
    assert np.isnan(npo.hard_cross_entropy(np.zeros((1, 5, 20, 20), np.float32), g["labels"])[0])


def test_soft_label_ce_golden(golden):
    g = golden("soft_ce")
    pred = torch.from_numpy(g["pred"]).requires_grad_(True)
    soft = torch.from_numpy(g["soft"])
    loss = to.soft_label_cross_entropy(pred, soft)
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < 1e-6
    np.testing.assert_allclose(pred.grad.numpy(), g["grad"], rtol=1e-5, atol=1e-9)
    assert abs(npo.soft_label_cross_entropy(g["pred"], g["soft"]) - float(g["loss"])) < 2e-6
    np.testing.assert_allclose(npo.soft_label_cross_entropy_grad(g["pred"], g["soft"]), g["grad"], rtol=1e-4, atol=1e-8)
    w = torch.from_numpy(g["weights"])
    assert abs(to.soft_label_cross_entropy(pred, soft, w).item() - float(g["loss_w"])) < 1e-6
    np.testing.assert_allclose(npo.soft_label_cross_entropy_grad(g["pred"], g["soft"], g["weights"]),
                               g["grad_w"], rtol=1e-4, atol=1e-8)


def test_discriminator_and_soft_label_builder_golden(golden):
    g = golden("discriminator")
    ncls = int(g["num_classes"])
    D = to.PixelDiscriminatorOracle(24, 16, num_classes=ncls)
    sd = {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")}
    assert list(sd.keys()) == list(D.state_dict().keys())
    D.load_state_dict(sd)
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        np.testing.assert_allclose(D(x).numpy(), g["out_lr"], rtol=1e-5, atol=1e-6)
        out_hr = D(x, (20, 27))
        np.testing.assert_allclose(out_hr.numpy(), g["out_hr"], rtol=1e-5, atol=1e-6)
        scaled = torch.from_numpy(g["seg_hr"]).div(1.8)
        q0 = to.build_soft_label(scaled, slot=0)
        q1 = to.build_soft_label(scaled, slot=1)
        # CPU softmax rounds the last bit differently from host to host (vector width, thread split): a few ulp, not bit for bit
        np.testing.assert_allclose(q0[:, :ncls].numpy(), g["soft"], rtol=1e-6, atol=0)
        np.testing.assert_allclose(q1[:, ncls:].numpy(), g["soft"], rtol=1e-6, atol=0)
        assert float(q0[:, ncls:].abs().max()) == 0.0 and float(q1[:, :ncls].abs().max()) == 0.0
        assert abs(to.soft_label_cross_entropy(out_hr, q0).item() - float(g["loss_slot0"])) < 1e-6
        assert abs(to.soft_label_cross_entropy(out_hr, q1).item() - float(g["loss_slot1"])) < 1e-6


def test_eval_golden(golden):
    g = golden("eval")
    ncls = int(g["num_classes"])
    head = _head_from_golden(g, g["f0.x"].shape[1], ncls)
    meter = to.AverageMeterOracle()
    cmt = torch.zeros(ncls, ncls, dtype=torch.int64)
    for f in range(3):
        x = torch.from_numpy(g[f"f{f}.x"])
        y = torch.from_numpy(g[f"f{f}.y"])
        pred, cm, (i, u, t, r) = to.eval_frame(head, x, y, ncls, literal_loop=True)
        np.testing.assert_array_equal(pred.numpy(), g[f"f{f}.pred"])
        np.testing.assert_array_equal(cm.numpy(), g[f"f{f}.cm"])
        cm_fast = to.confusion_matrix_bincount(ncls, pred.flatten(), y.flatten())
        np.testing.assert_array_equal(cm_fast.numpy(), g[f"f{f}.cm"])
        np.testing.assert_array_equal(npo.confusion_matrix(ncls, pred.numpy(), y.numpy()), g[f"f{f}.cm"])
        np.testing.assert_array_equal(npo.softmax_first_max(
            npo.upsample_bilinear_ac(g[f"f{f}.logits_lr"], y.shape[-2:])), g[f"f{f}.pred"])
        for got, key in ((i, "I"), (u, "U"), (t, "T"), (r, "R")):
            np.testing.assert_array_equal(got.numpy(), g[f"f{f}.{key}"])
        di, du, dt, do = npo.iutr_from_confusion(cm.numpy())
        np.testing.assert_array_equal(di, g[f"f{f}.I"]); np.testing.assert_array_equal(du, g[f"f{f}.U"])
        np.testing.assert_array_equal(dt, g[f"f{f}.T"]); np.testing.assert_array_equal(do, g[f"f{f}.R"])
        meter.update(i.numpy(), u.numpy(), t.numpy(), r.numpy())
        cmt = cmt + cm
    np.testing.assert_array_equal(cmt.numpy(), g["cmt"])
    np.testing.assert_allclose(meter.iou_sum, g["meter_iou_sum"], rtol=1e-6)
    np.testing.assert_allclose(meter.f1_sum, g["meter_f1_sum"], rtol=1e-6)
    np.testing.assert_array_equal(meter.intersection_sum, g["meter_intersection_sum"])
    np.testing.assert_array_equal(meter.union_sum, g["meter_union_sum"])


@pytest.mark.slow
def test_anchor_known_answer_full_size():
    """SURVEY.md section 8c anchor: seed-0, config-1 shapes, loss = 4.04814 (torch 2.11 CPU)."""
    torch.manual_seed(0)
    head = to.AsppHeadOracle(2048, RATES, RATES, 19)
    x = torch.randn(2, 2048, 65, 129)
    lab = torch.randint(0, 19, (2, 512, 1024))
    lab[torch.rand(2, 512, 1024) < 0.1] = 255
    with torch.no_grad():
        loss = to.hard_cross_entropy(head(x, (512, 1024)), lab)
    assert abs(loss.item() - 4.04814) < 5e-5


def _assert_state_dict_equal(module, g):
    sd = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    assert list(module.state_dict().keys()) == list(sd.keys())
    for k, v in module.state_dict().items():
        np.testing.assert_array_equal(v.numpy(), sd[k], err_msg=k)


@pytest.mark.parametrize("name,seed,cin,ncls", [("head_c19", 1, 24, 19), ("head_c2", 2, 16, 2), ("head_c19_T18", 3, 32, 19)])
def test_oracle_seeded_init_matches_reference_golden(golden, name, seed, cin, ncls):
    """Same seed, same init order as the reference (oracle/gen_golden.py seeds its modules the same way) => identical
    parameters; the seeded module then reproduces the reference's outputs (to the golden tolerance: CPU convolutions may
    round differently from machine to machine)."""
    g = golden(name)
    torch.manual_seed(seed)
    head = to.AsppHeadOracle(cin, RATES, RATES, ncls)
    _assert_state_dict_equal(head, g)
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        np.testing.assert_allclose(head(x, g["labels"].shape[-2:]).numpy(), g["logits_hr"], rtol=1e-5, atol=1e-6)


def test_discriminator_oracle_seeded_init_matches_reference_golden(golden):
    g = golden("discriminator")
    torch.manual_seed(21)
    D = to.PixelDiscriminatorOracle(24, 16, num_classes=int(g["num_classes"]))
    _assert_state_dict_equal(D, g)
    with torch.no_grad():
        np.testing.assert_allclose(D(torch.from_numpy(g["x"]), (20, 27)).numpy(), g["out_hr"], rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ 8f-3: test-time augmentation (flip / multi-scale)
class _Replay(torch.nn.Module):
    """Stands in for classifier(feature_extractor(.)): returns the recorded member logits in call order."""

    def __init__(self, outputs):
        super().__init__()
        self.outputs, self.k = outputs, 0

    def forward(self, feats, size=None):
        out = self.outputs[self.k]
        self.k += 1
        return out


def _assert_pred_equal_off_ties(probs, want_pred, gap=1e-6):
    top2 = probs.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > gap
    got = probs.max(1)[1]
    assert torch.equal(got[clear], torch.from_numpy(want_pred)[clear])
    assert float(clear.float().mean()) > 0.99


def test_tta_oracle_matches_reference_golden(golden):
    g = golden("tta")
    image, label = torch.from_numpy(g["image"]), torch.from_numpy(g["label"])
    size = label.shape[-2:]
    # inference(flip=True): the oracle's line-by-line restatement fed the recorded head outputs, and the from-members form
    both = torch.cat([torch.from_numpy(g["flip.member0"]), torch.from_numpy(g["flip.member1"])], 0)
    probs = to.inference(torch.nn.Identity(), _Replay([both]), image, label, flip=True)
    # CPU softmax rounds the last bit differently from host to host (vector width, thread split): a few ulp, not bit for bit
    np.testing.assert_allclose(probs.numpy(), g["flip.probs"], rtol=1e-6, atol=0)
    _assert_pred_equal_off_ties(probs, g["flip.pred"])
    # member by member the CPU kernels vectorise differently than on the batch of two: equal to an ulp, not bit for bit
    probs2 = to.tta_probabilities([both[0:1], both[1:2]], [False, True], size, divisors=(2,))
    np.testing.assert_allclose(probs2.numpy(), g["flip.probs"], rtol=1e-6, atol=1e-7)
    _assert_pred_equal_off_ties(probs2, g["flip.pred"])
    np.testing.assert_allclose(probs2.sum(1).numpy(), 1.0, atol=1e-5)
    # multi_scale_inference with and without flips
    for name, flip in (("ms", True), ("ms_noflip", False)):
        members = [torch.from_numpy(g[f"{name}.member{k}"]) for k in range(int(g[f"{name}.n_members"]))]
        scales = [float(s) for s in g["scales"]]
        probs = to.multi_scale_inference(torch.nn.Identity(), _Replay(members), image, label, flip=flip, scales=scales)
        np.testing.assert_allclose(probs.numpy(), g[f"{name}.probs"], rtol=1e-6, atol=0)
        _assert_pred_equal_off_ties(probs, g[f"{name}.pred"])
        flips = [bool(k % 2) for k in range(len(members))] if flip else [False] * len(members)
        probs2 = to.tta_probabilities(members, flips, size, divisors=(len(scales), 2) if flip else (len(scales),))
        np.testing.assert_allclose(probs2.numpy(), g[f"{name}.probs"], rtol=1e-6, atol=1e-7)
        _assert_pred_equal_off_ties(probs2, g[f"{name}.pred"])


def test_tta_oracle_end_to_end_matches_reference_golden(golden):
    """inference / multi_scale_inference driven through a backbone and head (rebuilt from the seeds oracle/gen_golden_tta.py
    used), so that the images the oracle feeds them -- mirrored, rescaled -- are checked too, not only the ensemble arithmetic."""
    g = golden("tta")
    torch.manual_seed(51)
    fe = torch.nn.Sequential(torch.nn.Conv2d(3, 12, 3, stride=4, padding=1), torch.nn.ReLU())
    head = to.AsppHeadOracle(12, RATES, RATES, int(g["num_classes"]))
    with torch.no_grad():
        for m in head.conv2d_list:
            m.weight.mul_(40.0)
    image, label = torch.from_numpy(g["image"]), torch.from_numpy(g["label"])
    scales = [float(s) for s in g["scales"]]
    for name, probs in (("flip", to.inference(fe, head, image, label, flip=True)),
                        ("ms", to.multi_scale_inference(fe, head, image, label, flip=True, scales=scales)),
                        ("ms_noflip", to.multi_scale_inference(fe, head, image, label, flip=False, scales=scales))):
        np.testing.assert_allclose(probs.numpy(), g[f"{name}.probs"], rtol=1e-5, atol=1e-6, err_msg=name)
        _assert_pred_equal_off_ties(probs, g[f"{name}.pred"], gap=1e-5)
    # the poly schedule itself is pinned by the reference's learning rates in optim.npz (test_optimizer_oracle_matches_reference_golden)
    with pytest.raises(NotImplementedError):
        to.adjust_learning_rate('step', 1.0, 1, 2, 0.9)


# ------------------------------------------------------------------ 8f-4: optimizer steps
def test_optimizer_oracle_matches_reference_golden(golden):
    g = golden("optim")
    n, steps = int(g["n"]), int(g["steps"])
    p0 = [torch.from_numpy(g[f"p0.{i}"]) for i in range(n)]
    grads = [[torch.from_numpy(g[f"g{k}.{i}"]) for i in range(n)] for k in range(steps)]
    lrs = [to.adjust_learning_rate('poly', float(g["base_lr"]), k, int(g["max_iter"]), float(g["power"])) for k in range(steps)]
    np.testing.assert_array_equal(np.asarray(lrs), g["lrs"])
    ps, st = to.optimizer_steps("sgd", p0, grads, lrs=[lr * 10 for lr in lrs], lr=lrs[0] * 10, momentum=0.9, weight_decay=5e-4)
    for i in range(n):
        np.testing.assert_array_equal(ps[i].numpy(), g[f"sgd.p.{i}"])
        np.testing.assert_array_equal(st[i][0].numpy(), g[f"sgd.buf.{i}"])
    ps, st = to.optimizer_steps("adam", p0, grads, lrs=[lr * 0.4 for lr in lrs], lr=1e-4, betas=(0.9, 0.99))
    for i in range(n):
        np.testing.assert_array_equal(ps[i].numpy(), g[f"adam.p.{i}"])
        np.testing.assert_array_equal(st[i][0].numpy(), g[f"adam.m.{i}"])
        np.testing.assert_array_equal(st[i][1].numpy(), g[f"adam.v.{i}"])


def test_fada_iteration_oracle_equals_fada_step_losses_and_moves_parameters():
    """The iteration with optimizer steps (aspp_fada.py:80-127) logs the same four losses as the step without them -- the head's
    step comes after its last use in the iteration, the discriminator's at the very end -- and leaves updated parameters."""
    import copy
    torch.manual_seed(3)
    head = to.AsppHeadOracle(8, RATES, RATES, 5)
    D = to.PixelDiscriminatorOracle(8, 8, num_classes=5)
    head2, D2 = copy.deepcopy(head), copy.deepcopy(D)
    src, tgt = torch.relu(torch.randn(1, 8, 6, 7)), torch.relu(torch.randn(1, 8, 6, 7))
    lab = torch.randint(0, 5, (1, 24, 28))
    lab[0, :3] = 255
    want = to.fada_step(head, D, src, tgt, lab)
    oc = torch.optim.SGD(head2.parameters(), lr=2.5e-3, momentum=0.9, weight_decay=5e-4)
    od = torch.optim.Adam(D2.parameters(), lr=1e-4, betas=(0.9, 0.99))
    got = to.fada_iteration(head2, D2, oc, od, src, tgt, lab)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    assert all(not torch.equal(p, q) for p, q in zip(head.parameters(), head2.parameters()))
    assert all(not torch.equal(p, q) for p, q in zip(D.parameters(), D2.parameters()))


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def test_numpy_optimizer_restatement_matches_reference_golden(golden):
    """np_oracle.sgd_step / adam_step (the formulas the CUDA kernels implement, term by term) against the parameters and states
    torch.optim produced under the reference's setup: 1e-6 relative, the bar the GPU tests hold the kernels to."""
    g = golden("optim")
    n, steps = int(g["n"]), int(g["steps"])
    lrs = [float(v) for v in g["lrs"]]
    for i in range(n):
        p, buf = g[f"p0.{i}"], None
        for k in range(steps):
            p, buf = npo.sgd_step(p, g[f"g{k}.{i}"], buf, lr=lrs[k] * 10, momentum=0.9, weight_decay=5e-4)
        assert _rel(p, g[f"sgd.p.{i}"]) <= 1e-6 and _rel(buf, g[f"sgd.buf.{i}"]) <= 1e-6
        p, m, v = g[f"p0.{i}"], np.zeros_like(g[f"p0.{i}"]), np.zeros_like(g[f"p0.{i}"])
        for k in range(steps):
            p, m, v = npo.adam_step(p, g[f"g{k}.{i}"], m, v, k + 1, lr=lrs[k] * 0.4, beta1=0.9, beta2=0.99)
        assert _rel(p, g[f"adam.p.{i}"]) <= 1e-6 and _rel(m, g[f"adam.m.{i}"]) <= 1e-6 and _rel(v, g[f"adam.v.{i}"]) <= 4e-6


def test_numpy_tta_restatement_matches_reference_golden(golden):
    g = golden("tta")
    size = g["label"].shape[-2:]
    both = [g["flip.member0"], g["flip.member1"]]
    np.testing.assert_allclose(npo.tta_probabilities(both, [False, True], size, (2,)), g["flip.probs"], rtol=2e-6, atol=2e-7)
    members = [g[f"ms.member{k}"] for k in range(int(g["ms.n_members"]))]
    got = npo.tta_probabilities(members, [bool(k % 2) for k in range(len(members))], size, (3, 2))
    np.testing.assert_allclose(got, g["ms.probs"], rtol=2e-6, atol=2e-7)
    top2 = np.sort(g["ms.probs"], axis=1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > 1e-6
    assert np.array_equal(got.argmax(1)[clear], g["ms.pred"][clear])
