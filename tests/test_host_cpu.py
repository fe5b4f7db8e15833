"""CPU-only tests: C-ABI library loads and exports every symbol include/b200seg.h declares, host logic of the
drop-in layer (factories, state_dict contract, install(), error behaviour without a GPU), and the N>1 host path
under gloo with world_size 2."""
import os
import re
import sys
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    from rnd_semantic_segmentation_b200 import _build_ext, _lib
    _build_ext.build()
    return _lib.load()


def test_library_exports_every_declared_symbol(built_lib):
    from rnd_semantic_segmentation_b200 import _lib
    header = open(os.path.join(ROOT, "include", "b200seg.h")).read()
    declared = set(re.findall(r"\b(b200seg_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(built_lib, name), name
    assert built_lib.b200seg_abi_version() == 1
    assert built_lib.b200seg_aspp_packed_rows(19, 4) == 640          # 33 taps x 19 classes -> 627 -> 640
    assert built_lib.b200seg_aspp_packed_rows(2, 4) == 128
    assert built_lib.b200seg_upsample_ce_workspace_bytes(2, 19, 65, 129, 512, 1024) > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback(built_lib):
    import rnd_semantic_segmentation_b200 as b200
    from rnd_semantic_segmentation_b200._lib import B200SegError
    assert built_lib.b200seg_device_sms() < 0
    assert b"no CUDA device" in built_lib.b200seg_last_error()
    head = b200.ASPP_Classifier_V2(16, [6, 12, 18, 24], [6, 12, 18, 24], 3)
    with pytest.raises(B200SegError):
        head(torch.randn(1, 16, 8, 8))
    with pytest.raises(B200SegError):
        b200.soft_label_cross_entropy(torch.randn(1, 4, 3, 3), torch.rand(1, 4, 3, 3))
    with pytest.raises(B200SegError):
        b200.upsample_cross_entropy(torch.randn(1, 4, 3, 3), torch.zeros(1, 6, 6, dtype=torch.int64))
    with pytest.raises(B200SegError):
        b200.confusion_matrix(4, torch.zeros(5, dtype=torch.int64), torch.zeros(5, dtype=torch.int64))
    # the discriminator's conv stack is ours too (K6): no cuDNN / CPU path behind it
    D = b200.PixelDiscriminator(16, 16, num_classes=3)
    with pytest.raises(B200SegError):
        D(torch.randn(1, 16, 8, 8))
    with pytest.raises(B200SegError):
        D.forward_soft_loss(torch.randn(1, 16, 8, 8), torch.randn(1, 3, 8, 8), (16, 16), slot=0)
    # test-time augmentation (K7) and the fused optimizer steps (K8): same rule
    label = torch.zeros(1, 16, 16, dtype=torch.int64)
    out = b200.inference(torch.nn.Identity(), lambda feats, size=None: feats, torch.randn(1, 3, 4, 4), label, flip=True)
    assert tuple(out.shape) == (1, 3, 16, 16)                   # lazy: nothing has run yet
    with pytest.raises(B200SegError):
        out.max(1)
    with pytest.raises(B200SegError):
        out.cpu()
    p = torch.nn.Parameter(torch.zeros(4))
    p.grad = torch.ones(4)
    for opt in (b200.FusedSGD([p], lr=0.1, momentum=0.9), b200.FusedAdam([p], lr=0.1)):
        with pytest.raises(B200SegError):
            opt.step()
    assert float(p.detach().sum()) == 0.0                       # nothing was updated on the way to the error
    assert b200.adjust_learning_rate('poly', 2.5e-4, 0, 100, 0.9) == 2.5e-4
    with pytest.raises(NotImplementedError):
        b200.adjust_learning_rate('cosine', 2.5e-4, 0, 100, 0.9)
    # C-ABI argument errors are reported, not crashed on, without a device
    assert built_lib.b200seg_tta_argmax_confusion(None, None, None, None, 2, 19, None, 8, 8, 255, None, 0, 0, None, None, None, None) != 0
    assert built_lib.b200seg_sgd_step(1, None, None, None, None, 0.1, 0.9, 0.0, 0.0, 0, 0, 1.0, None) != 0
    assert built_lib.b200seg_conv3x3_dgrad_colsum_scratch_bytes(4, 64, 128, 256) == 4 * 64 * 4 * 256 * 4
    assert built_lib.b200seg_conv3x3_wgrad_scratch_bytes(4, 64, 128, 256, 2048, 1) == 9 * 256 * 2048 * 4 + 256
    assert built_lib.b200seg_nhwc_colsum_scratch_bytes(256) > 0
    assert built_lib.b200seg_conv3x3_forward(None, 1, 8, 8, 16, 16, None, 16, 1, None, 0, 0.0, None, 16, None, None) != 0


def _cfg(name="deeplab_resnet101", C=19):
    return types.SimpleNamespace(MODEL=types.SimpleNamespace(NAME=name, NUM_CLASSES=C, WEIGHTS="", FREEZE_BN=True))


def test_factories_and_state_dict_contract():
    import rnd_semantic_segmentation_b200 as b200
    from oracle import torch_oracle as to
    torch.manual_seed(3)
    cls = b200.build_classifier(_cfg())
    torch.manual_seed(3)
    ref = to.AsppHeadOracle(2048, [6, 12, 18, 24], [6, 12, 18, 24], 19)
    assert list(cls.state_dict().keys()) == [f"conv2d_list.{i}.{p}" for i in range(4) for p in ("weight", "bias")]
    for (ka, va), (kb, vb) in zip(cls.state_dict().items(), ref.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)                         # same seed, same init order
    assert sum(p.numel() for p in cls.parameters()) == 1400908         # SURVEY section 8a
    assert b200.build_classifier(_cfg("deeplab_vgg16")).conv2d_list[0].in_channels == 1024
    with pytest.raises(NotImplementedError):
        b200.build_classifier(_cfg("deeplab_mobilenet"))
    D = b200.build_adversarial_discriminator(_cfg())
    assert list(D.state_dict().keys()) == ["D.0.weight", "D.0.bias", "D.2.weight", "D.2.bias", "cls1.weight", "cls1.bias",
                                           "cls2.weight", "cls2.bias"]
    assert sum(p.numel() for p in D.parameters()) == 5057702
    assert b200.build_adversarial_discriminator(_cfg("x_efficientnetb2")).D[0].in_channels == 1408
    assert b200.build_adversarial_discriminator(_cfg("x_hardnet68"), num_features=77).D[0].in_channels == 77
    with pytest.raises(NotImplementedError):
        b200.build_adversarial_discriminator(_cfg("deeplab_foo"))
    # reference-format checkpoint round trip incl. the 'module.' prefix DDP adds
    sd = {"module." + k: v for k, v in ref.state_dict().items()}
    cls.load_state_dict({k[len("module."):]: v for k, v in sd.items()})
    with pytest.raises(NotImplementedError):
        b200.ASPP_Classifier_V2(8, [6, 12], [1, 2], 3)._rates()


def test_average_meter_and_numpy_iou_match_oracle():
    import rnd_semantic_segmentation_b200 as b200
    from oracle import torch_oracle as to
    rng = np.random.RandomState(0)
    a, b = b200.AverageMeter(), to.AverageMeterOracle()
    for _ in range(4):
        pd = rng.randint(0, 5, (40, 50)); gt = rng.randint(0, 5, (40, 50)); gt[rng.rand(40, 50) < 0.2] = 255
        i, u, t, r = b200.intersectionAndUnion(pd, gt, 5)
        i2, u2, t2, r2 = to.intersection_and_union(torch.from_numpy(pd), torch.from_numpy(gt), 5)
        for x, y in ((i, i2), (u, u2), (t, t2), (r, r2)):
            np.testing.assert_array_equal(x, y.numpy().astype(np.int64))
        args = [v.astype(np.float32) for v in (i, u, t, r)]
        a.update(*args); b.update(*args)
    ra, rb = a.results(), b.results()
    for k in ("macro_iou", "macro_f1", "micro_iou", "micro_f1"):
        np.testing.assert_array_equal(ra[k], rb[k])


def test_install_patches_reference_modules(monkeypatch):
    import rnd_semantic_segmentation_b200 as b200
    core = types.ModuleType("core"); models = types.ModuleType("core.models"); bld = types.ModuleType("core.models.build")
    utils = types.ModuleType("core.utils"); util = types.ModuleType("core.utils.utility"); tester = types.ModuleType("core.testers.aspp_tester")
    bld.build_classifier = models.build_classifier = lambda cfg: "ref"
    util.confusion_matrix = tester.confusion_matrix = lambda *a: "ref"
    for m in (core, models, bld, utils, util, tester):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    patched = b200.install()
    assert bld.build_classifier is b200.build_classifier and models.build_classifier is b200.build_classifier
    assert util.confusion_matrix is b200.confusion_matrix and tester.confusion_matrix is b200.confusion_matrix
    assert "core.utils.utility.soft_label_cross_entropy" in patched
    assert util.multi_scale_inference is b200.multi_scale_inference and util.get_color_palette is b200.get_color_palette
    # optional: the trainers' torch.optim.SGD / Adam constructions build the fused subclasses for CUDA parameters only
    inst = sys.modules["rnd_semantic_segmentation_b200.install"]      # (the package attribute `install` is the function)
    stock_sgd, stock_adam = torch.optim.SGD, torch.optim.Adam
    try:
        assert "torch.optim.SGD" in b200.install(optimizers=True)
        cpu_opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(2))], lr=0.1, momentum=0.9)
        assert type(cpu_opt) is stock_sgd                       # CPU parameters keep the stock optimizer
        assert type(torch.optim.Adam([{"params": [torch.nn.Parameter(torch.zeros(2))]}], lr=0.1)) is stock_adam
    finally:
        inst.uninstall_optimizers()
    assert torch.optim.SGD is stock_sgd and torch.optim.Adam is stock_adam


def test_synth_shapes_and_determinism():
    from rnd_semantic_segmentation_b200 import synth
    lab = synth.make_labels(2, 100, 130, 19, seed=5)
    assert lab.shape == (2, 100, 130) and lab.dtype == torch.int64
    assert set(torch.unique(lab).tolist()) <= set(range(19)) | {255}
    assert torch.equal(lab, synth.make_labels(2, 100, 130, 19, seed=5))
    x = synth.make_features(1, 16, 5, 7, seed=2)
    assert float(x.min()) >= 0 and x.shape == (1, 16, 5, 7)
    assert synth.WORKLOADS["deeplabv2_r101_src"] == (2, 2048, 65, 129, 512, 1024, 19)


def _dist_worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    from rnd_semantic_segmentation_b200 import distributed as D
    import rnd_semantic_segmentation_b200 as b200
    assert D.init_from_env("gloo")
    # under a multi-rank process group module(x, size) defaults to the materialised tensor: the reference's
    # DistributedDataParallel(find_unused_parameters=True) wrapper (train_distill.py:54-62) looks for tensors in the output
    from rnd_semantic_segmentation_b200 import lazy
    assert lazy.lazy_enabled(None) is False and lazy.lazy_enabled(True) is True and lazy.lazy_enabled(False) is False
    torch.manual_seed(0)
    head = b200.ASPP_Classifier_V2(8, [6, 12, 18, 24], [6, 12, 18, 24], 3)
    assert head.lazy is None
    for i, p in enumerate(head.parameters()):
        p.grad = torch.full_like(p, float(rank + 1) * (i + 1))
    bucket = D.allreduce_mean_grads_(head)
    for i, p in enumerate(head.parameters()):
        assert torch.allclose(p.grad, torch.full_like(p, 1.5 * (i + 1)))       # mean of ranks (1, 2)
        assert p.grad.data_ptr() >= bucket.flat.data_ptr()
    # the discriminator's overlapped bucket (DDP semantics for the module train_adv.py never synchronises): .grad stays aliased to
    # the flat buffer across zero_grads_(), two backward passes accumulate in place, the mean lands in every rank's .grad, and the
    # optimizer step behind it leaves bit-identical parameters on all ranks
    torch.manual_seed(1)
    model_D = b200.PixelDiscriminator(8, 8, num_classes=3)
    dbucket = D.OverlappedGradBucket(model_D.parameters())
    opt = torch.optim.Adam(model_D.parameters(), lr=1e-2, betas=(0.9, 0.99))
    for it in range(2):
        dbucket.zero_grads_()
        for k in range(2):                                  # two backward passes into the same gradients (aspp_fada.py:119-125)
            loss = sum(((p * float(rank + 1 + k + it)) ** 2).sum() for p in model_D.parameters())
            loss.backward()
        local = [p.grad.clone() for p in model_D.parameters()]
        assert all(p.grad.data_ptr() == v.data_ptr() for p, v in zip(dbucket.params, dbucket.views))
        dbucket.begin_allreduce_()
        dbucket.step(opt)
        dbucket.wait()
        gathered = [[torch.empty_like(g) for _ in range(world)] for g in local]
        for g, out in zip(local, gathered):
            torch.distributed.all_gather(out, g)
        for p, out in zip(model_D.parameters(), gathered):
            assert torch.allclose(p.grad, sum(out) / world, rtol=1e-6, atol=0)
    flat_params = torch.cat([p.detach().reshape(-1) for p in model_D.parameters()])
    both = [torch.empty_like(flat_params) for _ in range(world)]
    torch.distributed.all_gather(both, flat_params)
    assert torch.equal(both[0], both[1])
    # eval sharding: frames rank::world, int64 confusion matrix summed exactly
    frames = D.shard_indices(7, rank, world)
    cm = torch.zeros(3, 3, dtype=torch.int64)
    for f in frames:
        cm[f % 3, (f * 2) % 3] += 10 ** 12 + f            # beyond fp32/fp64-exact accumulation if done in float32
    D.allreduce_confusion_(cm)
    want = torch.zeros(3, 3, dtype=torch.int64)
    for f in range(7):
        want[f % 3, (f * 2) % 3] += 10 ** 12 + f
    assert torch.equal(cm, want)
    # macro metrics: per-frame areas gathered in frame order (7 frames over 2 ranks: shards of 4 and 3)
    local = torch.stack([torch.full((4, 3), f, dtype=torch.int64) + torch.arange(4).view(4, 1) for f in frames])
    areas = D.allgather_frame_areas(local, 7)
    assert tuple(areas.shape) == (7, 4, 3)
    for f in range(7):
        assert torch.equal(areas[f], torch.full((4, 3), f, dtype=torch.int64) + torch.arange(4).view(4, 1))
    torch.save(cm, os.path.join(tmp, f"cm{rank}.pt"))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def test_distributed_gloo_world2(tmp_path):
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_dist_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a, b = torch.load(tmp_path / "cm0.pt"), torch.load(tmp_path / "cm1.pt")
    assert torch.equal(a, b)


def test_color_palette_png_round_trip(tmp_path):
    """get_color_palette (utility.py:211-217: Image.fromarray(pred.astype('uint8')).convert('P'), putpalette(palette)): a mode-'P'
    image whose indices are the label ids and whose palette is the given one, all 256 entries of it."""
    import rnd_semantic_segmentation_b200 as b200
    from PIL import Image
    rng = np.random.default_rng(0)
    pred = rng.integers(0, 19, size=(37, 53)).astype(np.int64)
    palette = [int(v) for v in rng.integers(0, 256, size=19 * 3)] + [0] * (256 * 3 - 19 * 3)
    img = b200.get_color_palette(pred, palette)
    assert img.mode == "P" and img.size == (53, 37) and img.palette.mode == "RGB"
    np.testing.assert_array_equal(np.asarray(img), pred.astype(np.uint8))
    assert img.getpalette() == palette
    path = tmp_path / "mask.png"
    img.save(path)
    back = Image.open(path)
    np.testing.assert_array_equal(np.asarray(back), pred.astype(np.uint8))
    np.testing.assert_array_equal(np.asarray(back.convert("RGB")), np.asarray(palette[:57], dtype=np.uint8).reshape(19, 3)[pred])


def test_fused_optimizers_pickle_and_state_dict_contract():
    """FusedSGD / FusedAdam are torch.optim.SGD / Adam for everything but step(): identical state_dict layout (the reference's
    checkpoints hold optimizer_cls / optimizer_D state dicts, aspp_trainer.py:46-55), picklable / deep-copyable with the gradient
    scale kept and no launch plan (raw pointers) carried over."""
    import copy
    import pickle
    import rnd_semantic_segmentation_b200 as b200
    ps = [torch.nn.Parameter(torch.zeros(3)), torch.nn.Parameter(torch.zeros(2, 2))]
    pairs = ((b200.FusedSGD(ps, lr=0.1, momentum=0.9, weight_decay=5e-4, grad_scale=0.125), torch.optim.SGD(ps, lr=0.1, momentum=0.9, weight_decay=5e-4)),
             (b200.FusedAdam(ps, lr=1e-4, betas=(0.9, 0.99)), torch.optim.Adam(ps, lr=1e-4, betas=(0.9, 0.99))))
    for ours, stock in pairs:
        assert isinstance(ours, type(stock))
        a, b = ours.state_dict(), stock.state_dict()
        assert a["param_groups"] == b["param_groups"] and a["state"] == b["state"]
        stock.load_state_dict(a)
        ours.load_state_dict(b)
        ours._plans[0] = {"ids": []}
        for clone in (copy.deepcopy(ours), pickle.loads(pickle.dumps(ours))):
            assert type(clone) is type(ours) and clone._plans == {} and clone.grad_scale == ours.grad_scale
            assert clone.state_dict()["param_groups"] == a["param_groups"]


def test_c_side_split_rule_matches_the_python_one(built_lib):
    """b200seg_head_loss_backward picks the weight-gradient split-K factor itself; it must be the rule the separate entries use."""
    from rnd_semantic_segmentation_b200 import _lib
    lib = _lib.load()
    for P in (1, 63, 64, 200, 1936, 8385, 16770, 30976, 67080, 131072, 1 << 22):
        for C, Cin, R in ((19, 2048, 4), (2, 2048, 4), (19, 256, 4), (7, 64, 2), (32, 512, 1)):
            assert lib.b200seg_aspp_default_wgrad_splits(P, C, Cin, R) == _lib.default_wgrad_splits(P, C, Cin, R), (P, C, Cin, R)
    assert lib.b200seg_head_loss_workspace_bytes(2, 2048, 19, 65, 129, 4, 512, 1024, 0) > 2 * 65 * 129 * 2048 * 2
    assert lib.b200seg_head_loss_workspace_bytes(2, 2048, 19, 65, 129, 4, 512, 1024, 1) < 2 * 65 * 129 * 2048 * 2
    assert lib.b200seg_head_loss_workspace_bytes(0, 2048, 19, 65, 129, 4, 512, 1024, 0) == 0


def test_lazy_logits_default_is_automatic():
    """Single process, no process group: lazy; B200SEG_LAZY overrides; an explicit module attribute overrides both."""
    from rnd_semantic_segmentation_b200 import lazy
    old = os.environ.pop("B200SEG_LAZY", None)
    try:
        assert lazy.lazy_enabled(None) is True
        os.environ["B200SEG_LAZY"] = "0"
        assert lazy.lazy_enabled(None) is False and lazy.lazy_enabled(True) is True
        os.environ["B200SEG_LAZY"] = "1"
        assert lazy.lazy_enabled(None) is True and lazy.lazy_enabled(False) is False
    finally:
        os.environ.pop("B200SEG_LAZY", None)
        if old is not None:
            os.environ["B200SEG_LAZY"] = old


def test_public_header_is_plain_c(tmp_path):
    """include/b200seg.h is the drop-in boundary: it must compile as C99 and as C++ on its own (no torch / CUDA types), and a C
    program that only includes it and calls a host-side query must link against libb200seg.so."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    hdr = os.path.join(ROOT, "include", "b200seg.h")
    subprocess.run(["gcc", "-fsyntax-only", "-x", "c", "-std=c99", "-Wall", "-Werror", hdr], check=True)
    subprocess.run(["g++", "-fsyntax-only", "-x", "c++", "-Wall", "-Werror", hdr], check=True)
    from rnd_semantic_segmentation_b200 import _build_ext
    so = _build_ext.build()
    src = tmp_path / "t.c"
    src.write_text('#include <stdio.h>\n#include "b200seg.h"\nint main(void) {\n'
                   '  printf("%d %d %d\\n", b200seg_abi_version(), b200seg_aspp_packed_rows(19, 4), b200seg_aspp_default_wgrad_splits(67080, 19, 2048, 4));\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "t"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), so,
                    "-Wl,-rpath," + os.path.dirname(so)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert out == ["1", "640", "6"], out
