"""The seam-format tail with batch statistics: the last Bottleneck's bn3 as a training-mode BatchNorm2d / SyncBatchNorm
(statistics, running-statistics update, SyncBatchNorm exchange, forward and backward), fuse_backbone_tail(train_bn=True) and
install(seam=True, seam_train_bn=True).

PyTorch's own batch-norm ops (torch.batch_norm_stats, torch.batch_norm_gather_stats_with_counts, torch.batch_norm_backward_reduce,
torch.batch_norm_backward_elemt -- what SyncBatchNorm is built from) and fp64 statistics are the references; an R-rank
SyncBatchNorm is emulated on one GPU by sharding the batch.  The blocks are test_seam_tail.py's restated Bottleneck."""
import copy
import datetime
import inspect
import sys
import types

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import rel_err
from test_seam_tail import _block_and_head, _check_train_bars, _train_step, make_block, same

import rnd_semantic_segmentation_b200 as b200
from rnd_semantic_segmentation_b200 import seam


def _train_bn_block(seed=31, momentum=0.1):
    blk = make_block(64, 16, seed, norm=nn.BatchNorm2d).train()
    for m in blk.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.momentum = momentum
    return blk


# ------------------------------------------------------------------ CPU: opt-in flag, kind table, install()
@pytest.mark.parametrize("momentum", [0.1, None])
def test_training_batchnorm_block_cpu_forward_matches_unfused(momentum):
    blk = _train_bn_block(momentum=momentum)
    ref = copy.deepcopy(blk)
    b200.fuse_backbone_tail(nn.Sequential(blk), train_bn=True)
    assert blk.__dict__["forward"].train_bn
    x = torch.randn(2, 64, 9, 13)
    for _ in range(3):
        out, want = blk(x), ref(x)
        assert out.dtype == torch.float32 and torch.equal(out, want)
    with torch.no_grad():
        assert torch.equal(blk(x), ref(x))
    for a, b in ((blk.bn3.running_mean, ref.bn3.running_mean), (blk.bn3.running_var, ref.bn3.running_var),
                 (blk.bn3.num_batches_tracked, ref.bn3.num_batches_tracked)):
        assert torch.equal(a, b)
    assert int(blk.bn3.num_batches_tracked) == 4


def test_train_bn_flag_survives_save_load_and_deepcopy_and_follows_repeated_calls(tmp_path):
    fe = nn.Sequential(_train_bn_block())
    b200.fuse_backbone_tail(fe, train_bn=True)
    path = tmp_path / "fe.pt"
    torch.save(fe, path)
    loaded = torch.load(path, weights_only=False)
    assert seam.is_fused(loaded) and loaded[0].__dict__["forward"].train_bn
    clone = copy.deepcopy(fe)
    assert clone[0].__dict__["forward"].train_bn and clone[0].__dict__["forward"].block is clone[0]
    b200.fuse_backbone_tail(fe)                                   # a repeated call with another value updates the flag
    assert not fe[0].__dict__["forward"].train_bn
    b200.fuse_backbone_tail(fe, train_bn=True)
    assert fe[0].__dict__["forward"].train_bn
    plain = nn.Sequential(_train_bn_block())
    b200.fuse_backbone_tail(plain)
    assert not plain[0].__dict__["forward"].train_bn


def test_norm_kind_table_with_train_bn():
    class SubBN(nn.BatchNorm2d):
        pass

    bn, sbn = nn.BatchNorm2d(16), nn.SyncBatchNorm(16)
    assert seam._norm_kind(bn) is None and seam._norm_kind(sbn) is None          # default: unchanged
    assert seam._norm_kind(bn, True) == "batch" and seam._norm_kind(sbn, True) == "batch"
    assert seam._norm_kind(SubBN(16), True) is None
    assert seam._norm_kind(nn.BatchNorm2d(16, track_running_stats=False), True) is None
    assert seam._norm_kind(nn.BatchNorm2d(16, affine=False), True) == "batch"
    sbn.eval()
    assert seam._norm_kind(sbn) is None
    assert seam._norm_kind(sbn, True) is None                                   # eval, but weight / bias want a gradient
    sbn.requires_grad_(False)
    assert seam._norm_kind(sbn, True) == "bn"
    scale, bias = seam._fold(sbn, "bn")
    assert seam._probe_ok(sbn, "bn", scale, bias)
    bn.eval().requires_grad_(False)
    assert seam._norm_kind(bn, True) == "bn"                                    # eval BatchNorm2d: the fold, as before


def test_install_seam_train_bn_wraps_the_factory_with_the_flag(monkeypatch):
    core = types.ModuleType("core"); models = types.ModuleType("core.models"); bld = types.ModuleType("core.models.build")

    def build_feature_extractor(cfg):
        return nn.Sequential(_train_bn_block())

    bld.build_feature_extractor = models.build_feature_extractor = build_feature_extractor
    bld.build_classifier = models.build_classifier = lambda cfg: "ref"
    for m in (core, models, bld):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    b200.install(seam=True)
    fn = bld.build_feature_extractor
    fe = fn(None)
    assert seam.is_fused(fe) and not fe[0].__dict__["forward"].train_bn            # training BN stays stock
    b200.install(seam=True, seam_train_bn=True)
    assert bld.build_feature_extractor is fn and models.build_feature_extractor is fn
    assert inspect.signature(fn) == inspect.signature(build_feature_extractor)
    assert fn(None)[0].__dict__["forward"].train_bn
    b200.install(seam=True)
    assert not fn(None)[0].__dict__["forward"].train_bn


# ------------------------------------------------------------------ GPU: statistics and combine
def _stats_input(shape, seed, unaligned=False, nan=False, special=True):
    N, C, h, w = shape
    g = torch.Generator().manual_seed(seed)
    c = 0.5 * torch.randn(N, C, h, w, generator=g) + torch.randn(1, C, 1, 1, generator=g)
    if special:
        c[:, 0] = 1e3 + 1.0 * torch.randn(N, h, w, generator=g)      # mean = 10^3 sigma
        c[:, 1] = 3.25                                               # constant: variance 0
    if nan:
        c[N - 1, 2, h - 1, w - 1] = float("nan")
    c = c.cuda()
    if unaligned:                                                    # a base 4 bytes past a 16-byte boundary
        flat = torch.empty(c.numel() + 1, device="cuda")
        flat[1:] = c.flatten()
        c = flat[1:].view(N, C, h, w)
    return c


STAT_SHAPES = [((8, 2048, 64, 128), False), ((2, 40, 65, 129), False), ((2, 64, 44, 44), False), ((3, 32, 9, 13), False),
               ((2, 16, 9, 13), True), ((1, 64, 33, 65), False), ((1, 64, 32, 64), True)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,unaligned", STAT_SHAPES)
def test_batch_statistics_against_fp64_and_torch(shape, unaligned):
    from rnd_semantic_segmentation_b200 import _lib
    c = _stats_input(shape, 1, unaligned=unaligned, nan=True)
    assert (c.data_ptr() % 16 != 0) == unaligned
    rec = _lib.bn_stats(c)
    assert same(_lib.bn_stats(c), rec)                               # fixed reduction order: bit-identical
    M = shape[0] * shape[2] * shape[3]
    assert torch.all(rec[0] == M)
    mean, var = rec[1], rec[2] / M
    cd = c.double()
    want_mean, want_var = cd.mean((0, 2, 3)), cd.var((0, 2, 3), unbiased=False)
    nan = torch.isnan(want_mean)
    assert nan.tolist() == torch.isnan(mean).tolist() == torch.isnan(var).tolist() and int(nan.sum()) == 1 and bool(nan[2])
    ok = ~nan
    sigma = want_var.sqrt()
    assert torch.all((mean - want_mean).abs()[ok] <= 1e-6 * (want_mean.abs() + sigma)[ok])
    assert torch.all((var - want_var).abs()[ok] <= 1e-5 * want_var[ok])
    assert var[1].item() == 0.0
    eps = 1e-5
    m32, inv32, count = _lib.bn_combine_stats(rec, eps)
    assert count.item() == M
    tm, tinv = torch.batch_norm_stats(c, eps)
    assert torch.isnan(m32[2]) and torch.isnan(inv32[2])
    assert torch.all((m32.double() - tm.double()).abs()[ok] <= 1e-6 * (want_mean.abs() + sigma)[ok])
    # (PyTorch's fp32 Welford loses more than we do on the 10^3-sigma channel; fp64 below is the tight reference)
    assert torch.all(((inv32.double() - tinv.double()).abs() / tinv.double())[ok] <= 1e-4)
    assert torch.all(((inv32.double() - (want_var + eps).rsqrt()).abs() / (want_var + eps).rsqrt())[ok] <= 1e-6)


def _rel(a, b):
    """Largest element-wise relative difference (for quantities bounded away from 0: invstd)."""
    return ((a.double() - b.double()).abs() / b.double().abs().clamp_min(1e-30)).max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("splits", [[7], [3, 4], [1, 2, 1, 3]])
@pytest.mark.parametrize("momentum", [0.1, None])
def test_combine_of_rank_records_matches_gather_stats_with_counts(splits, momentum):
    from rnd_semantic_segmentation_b200 import _lib
    C, eps = 96, 1e-5
    c = _stats_input((sum(splits), C, 17, 23), 2, special=False)
    shards = list(torch.split(c, splits))
    g = torch.Generator().manual_seed(3)
    rm0, rv0 = 0.1 * torch.randn(C, generator=g).cuda(), 0.5 + torch.rand(C, generator=g).cuda()
    nbt = torch.tensor(4, dtype=torch.int64, device="cuda")
    f = 1.0 / 4 if momentum is None else momentum
    records = torch.stack([_lib.bn_stats(s.contiguous()) for s in shards])
    rm, rv = rm0.clone(), rv0.clone()
    mean, invstd, count = _lib.bn_combine_stats(records, eps, momentum, rm, rv, nbt)
    stats = [torch.batch_norm_stats(s.contiguous(), eps) for s in shards]
    counts = torch.tensor([s.shape[0] * s.shape[2] * s.shape[3] for s in shards], dtype=torch.float32, device="cuda")
    trm, trv = rm0.clone(), rv0.clone()
    tmean, tinv = torch.batch_norm_gather_stats_with_counts(c, torch.stack([m for m, _ in stats]), torch.stack([i for _, i in stats]),
                                                            trm, trv, f, eps, counts)
    assert count.item() == counts.sum().item()
    scale = c.double().std((0, 2, 3)) + c.double().mean((0, 2, 3)).abs()
    assert ((mean.double() - tmean.double()).abs() / scale).max().item() <= 1e-6
    assert _rel(invstd, tinv) <= 1e-6
    # running buffers: max-abs over max-abs (a running mean near 0 has no element-wise relative scale)
    assert rel_err(rm, trm) <= 1e-6 and rel_err(rv, trv) <= 1e-6
    whole, whole_inv, _ = _lib.bn_combine_stats(_lib.bn_stats(c), eps)                  # the unsharded batch
    assert ((mean.double() - whole.double()).abs() / scale).max().item() <= 1e-6
    assert _rel(invstd, whole_inv) <= 1e-6


# ------------------------------------------------------------------ GPU: forward and backward kernels
def _tail_inputs(shape, seed, affine=True):
    N, C, h, w = shape
    g = torch.Generator().manual_seed(seed)
    c = (0.7 * torch.randn(N, C, h, w, generator=g) + 0.3 * torch.randn(1, C, 1, 1, generator=g)).cuda()
    identity = torch.randn(N, C, h, w, generator=g).cuda()
    weight = (0.5 + torch.rand(C, generator=g)).cuda() if affine else None
    bias = (0.2 * torch.randn(C, generator=g)).cuda() if affine else None
    return c, identity, weight, bias


def _within_one_bf16_ulp(a, b):
    """|a - b| <= one bf16 ulp of max(|a|, |b|); around 0, where relu follows a cancelling sum, 1e-6 absolute."""
    a, b = a.float(), b.float()
    m = torch.maximum(a.abs(), b.abs())
    ulp = torch.exp2(torch.floor(torch.log2(m.clamp_min(1e-30))) - 7)
    return bool(((a - b).abs() <= torch.maximum(ulp, torch.full_like(ulp, 1e-6))).all())


@pytest.mark.gpu
@pytest.mark.parametrize("shape,affine", [((8, 2048, 64, 128), True), ((2, 40, 65, 129), True), ((2, 64, 9, 13), False)])
def test_forward_within_one_bf16_ulp_of_the_stock_block(shape, affine):
    c, identity, weight, bias = _tail_inputs(shape, 5, affine)
    C = shape[1]
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    y = b200.seam_tail_bn(c, identity, weight, bias, rm, rv, nbt, 0.1, 1e-5)
    srm, srv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    want = torch.relu(F.batch_norm(c, srm, srv, weight, bias, True, 0.1, 1e-5) + identity).to(torch.bfloat16)
    assert y.dtype == torch.bfloat16 and y.is_contiguous(memory_format=torch.channels_last)
    assert _within_one_bf16_ulp(y, want)
    n_diff = int((y != want).sum().item())
    print(f"batch-statistics tail {shape}: {n_diff} of {want.numel()} features differ from the stock output cast to bf16")
    assert n_diff < 2e-4 * want.numel()
    assert int(nbt) == 1 and rel_err(rm, srm) <= 1e-6 and rel_err(rv, srv) <= 1e-6


def _bn_backward_reference(dy, y, c, mean, invstd, weight, counts, shards):
    """torch.batch_norm_backward_reduce per shard, summed in rank order, then torch.batch_norm_backward_elemt per shard."""
    g = torch.where(y > 0, dy.float(), 0.0).contiguous()
    affine = weight is not None
    parts = [torch.batch_norm_backward_reduce(gs.contiguous(), cs.contiguous(), mean, invstd, weight, True, affine, affine)
             for gs, cs in zip(torch.split(g, shards), torch.split(c, shards))]
    sum_dy, sum_dy_xmu = parts[0][0], parts[0][1]
    for p in parts[1:]:
        sum_dy, sum_dy_xmu = sum_dy + p[0], sum_dy_xmu + p[1]
    dc = torch.cat([torch.batch_norm_backward_elemt(gs.contiguous(), cs.contiguous(), mean, invstd, weight, sum_dy, sum_dy_xmu, counts)
                    for gs, cs in zip(torch.split(g, shards), torch.split(c, shards))])
    return g, dc, parts


@pytest.mark.gpu
@pytest.mark.parametrize("shape,affine", [((8, 2048, 64, 128), True), ((2, 40, 65, 129), True), ((2, 64, 9, 13), False)])
def test_backward_against_torch_batch_norm_backward(shape, affine):
    from rnd_semantic_segmentation_b200 import _lib
    c, identity, weight, bias = _tail_inputs(shape, 6, affine)
    mean, invstd, count = _lib.bn_combine_stats(_lib.bn_stats(c), 1e-5)
    y = _lib.seam_tail_bn_forward(c, identity, mean, invstd, weight, bias)
    gen = torch.Generator().manual_seed(7)
    dy = torch.randn(shape, generator=gen).cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    counts = torch.tensor([shape[0] * shape[2] * shape[3]], dtype=torch.int32, device="cuda")
    g, want_dc, parts = _bn_backward_reference(dy, y, c, mean, invstd, weight, counts, [shape[0]])
    sums, gw, gb = _lib.seam_tail_bn_backward_reduce(dy, y, c, mean, invstd, affine, affine)
    dc, di = _lib.seam_tail_bn_backward(dy, y, c, mean, invstd, weight, sums, count)
    assert torch.equal(di, g)
    assert rel_err(dc, want_dc) <= 1e-5
    assert rel_err(sums[0], parts[0][0]) <= 1e-5 and rel_err(sums[1], parts[0][1]) <= 1e-5
    if affine:
        assert rel_err(gw, parts[0][2]) <= 1e-5 and rel_err(gb, parts[0][3]) <= 1e-5
    # through autograd: c, identity, weight and bias get their gradients
    ca, ia = c.clone().requires_grad_(True), identity.clone().requires_grad_(True)
    wa = None if weight is None else weight.clone().requires_grad_(True)
    ba = None if bias is None else bias.clone().requires_grad_(True)
    b200.seam_tail_bn(ca, ia, wa, ba, None, None, None, 0.1, 1e-5).backward(dy)
    assert torch.equal(ia.grad, g) and torch.equal(ca.grad, dc)
    if affine:
        assert torch.equal(wa.grad, gw) and torch.equal(ba.grad, gb)


@pytest.mark.gpu
@pytest.mark.parametrize("shards", [[2, 2], [1, 2, 1, 1]])
def test_sharded_backward_emulates_syncbatchnorm(shards):
    from rnd_semantic_segmentation_b200 import _lib
    shape = (sum(shards), 64, 33, 65)
    c, identity, weight, bias = _tail_inputs(shape, 8)
    cs = [t.contiguous() for t in torch.split(c, shards)]
    mean, invstd, count = _lib.bn_combine_stats(torch.stack([_lib.bn_stats(t) for t in cs]), 1e-5)
    y = _lib.seam_tail_bn_forward(c, identity, mean, invstd, weight, bias)
    gen = torch.Generator().manual_seed(9)
    dy = torch.randn(shape, generator=gen).cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    counts = torch.tensor([s * shape[2] * shape[3] for s in shards], dtype=torch.int32, device="cuda")
    _, want_dc, _ = _bn_backward_reference(dy, y, c, mean, invstd, weight, counts, shards)
    ys, dys = torch.split(y, shards), torch.split(dy, shards)
    sums = torch.stack([_lib.seam_tail_bn_backward_reduce(d, t, ct, mean, invstd)[0] for d, t, ct in zip(dys, ys, cs)])
    dc = torch.cat([_lib.seam_tail_bn_backward(d, t, ct, mean, invstd, weight, sums, count)[0] for d, t, ct in zip(dys, ys, cs)])
    assert rel_err(dc, want_dc) <= 1e-5


# ------------------------------------------------------------------ GPU: block + head, graph capture
@pytest.mark.gpu
@pytest.mark.parametrize("momentum", [0.1, None])
def test_training_batchnorm_block_plus_head_matches_stock(momentum):
    blk, head, x, labels = _block_and_head(norm=nn.BatchNorm2d)
    blk.train()
    for m in blk.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.momentum = momentum
    ref = copy.deepcopy(blk)
    b200.fuse_backbone_tail(nn.Sequential(blk), train_bn=True)
    for step in range(3):
        stock = _train_step(ref, head, x, labels)
        fused = _train_step(blk, head, x, labels)
        assert fused["feat"].dtype == torch.bfloat16                     # the batch-statistics kernels ran
        if step == 0:
            want = stock["feat"].to(torch.bfloat16)
            n_diff = int((fused["feat"] != want).sum().item())
            print(f"training-mode BatchNorm2d tail: {n_diff} of {want.numel()} features differ from the stock output cast to bf16")
            # about 270 of 8.8 M features (3e-5) one bf16 ulp from stock moved the head's weight gradient by 2.3e-5 of its largest
            # entry on a B200 (the eval-mode fold: 115 features, 2.7e-6); 5e-5 holds that with margin, well inside what the
            # forward test's 2e-4 budget of differing features would allow
            _check_train_bars(stock, fused, head_tol=5e-5)
    assert rel_err(blk.bn3.running_mean, ref.bn3.running_mean) <= 1e-6
    assert rel_err(blk.bn3.running_var, ref.bn3.running_var) <= 1e-6
    assert torch.equal(blk.bn3.num_batches_tracked, ref.bn3.num_batches_tracked)


@pytest.mark.gpu
@pytest.mark.parametrize("momentum", [0.1, None])
def test_graph_capture_replays_bit_identical_to_eager(momentum):
    shape = (2, 256, 33, 65)
    c0, id0, w0, b0 = _tail_inputs(shape, 10)
    c, identity = c0.clone().requires_grad_(True), id0.clone().requires_grad_(True)
    weight, bias = w0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    C = shape[1]
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    gen = torch.Generator().manual_seed(11)
    dy = torch.randn(shape, generator=gen).cuda().to(torch.bfloat16).contiguous(memory_format=torch.channels_last)

    def step():
        y = b200.seam_tail_bn(c, identity, weight, bias, rm, rv, nbt, momentum, 1e-5)
        return (y,) + torch.autograd.grad(y, (c, identity, weight, bias), dy)

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
    eager = step()
    for a, b in zip(replayed, eager):
        assert torch.equal(a, b)
    for a, b in zip(state1, (rm, rv, nbt)):
        assert torch.equal(a, b)
    eager_twice = step()
    reset()
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    assert int(nbt) == int(state0[2]) + 2
    assert torch.equal(static[0], eager_twice[0])
    eager_state = [t.clone() for t in (rm, rv)]
    reset()
    step()
    step()
    assert torch.equal(eager_state[0], rm) and torch.equal(eager_state[1], rv)


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
        b200.fuse_backbone_tail(fused, train_bn=True)
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
                             gb=bn3.bias.grad.clone())
        s, f = out["stock"], out["fused"]
        assert f["feat"].dtype == torch.bfloat16
        assert abs(f["loss"].item() - s["loss"].item()) <= 1e-6 * abs(s["loss"].item())
        assert max(rel_err(a, b) for a, b in zip(f["head"], s["head"])) <= 5e-5
        assert rel_err(f["x"], s["x"]) <= 2.0 ** -8
        for n, gs in s["params"].items():
            assert ((f["params"][n].double() - gs.double()).norm() / gs.double().norm()).item() <= 2.0 ** -8, n
        assert rel_err(f["rm"], s["rm"]) <= 1e-6 and rel_err(f["rv"], s["rv"]) <= 1e-6
        # identical on both ranks: the statistics (hence the running buffers) and, after DDP, the bn3 gradients
        for key in ("rm", "rv", "gw", "gb"):
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
