"""-m gpu: the ASPP head and the fused conv3 tail under every GEMM switch setting (b200seg_gemm_set_sharing / _dgrad_mode /
_fwd_mode / _narrow_tiles), one switch at a time from the default.  profiles/ measures A/B results with these switches, so each
setting must compute what the default computes: the same-rounding oracle bar of test_k1_head_forward_backward, the forward and
the data gradient (no split-K) bit for bit equal to the default run, the weight gradient (whose split count follows the
geometry) within fp32 reordering of it."""
import pytest
import torch

from helpers import RATES, bf16_round, effective_bf16_head, rel_err
from oracle import torch_oracle as to
from test_gemm_layouts import set_switches
from test_seam_conv3 import _check_against_oracle, _op_inputs

pytestmark = pytest.mark.gpu
TOL = 1e-3
WGRAD_REORDER = 1e-5          # max-abs / max-abs between two fp32 split-K orders of the weight gradient

SETTINGS = {
    "default": {},
    "sharing0": dict(sharing=0),              # one CTA per tile: 224 / 192-column tiles and the rows epilogue in them
    "sharing3": dict(sharing=3),
    "sharing4": dict(sharing=4),
    "sharing5": dict(sharing=5),              # no cta_group::2: the pixel-major GEMMs on multicast-B pairs (generic kernel)
    "dgrad0": dict(dgrad=0),
    "dgrad2": dict(dgrad=2),
    "fwd0": dict(fwd=0),
    "narrow0": dict(narrow=0),
    "sharing0-narrow0": dict(sharing=0, narrow=0),
    "sharing5-dgrad2": dict(sharing=5, dgrad=2),
}
DEFAULT = dict(sharing=1, narrow=1, dgrad=1, fwd=1)
# (n, Cin, C, h, w): the bench head; the data gradient's last N-tile 64 columns wide (Cin = 320); 8 columns (264); P = 128 (one M-tile)
SHAPES = [(2, 2048, 19, 33, 65), (1, 320, 19, 17, 23), (2, 264, 19, 9, 13), (1, 64, 19, 8, 16)]


@pytest.fixture(scope="module")
def lib():
    from rnd_semantic_segmentation_b200 import _lib
    _lib.load()
    yield _lib
    set_switches(_lib)


_ORACLE, _DEFAULT = {}, {}


def _head(shape):
    """(oracle head with the CUDA head's bf16 roundings, CUDA head, x, grad_output, oracle output, oracle grads) -- once per shape."""
    if shape not in _ORACLE:
        n, cin, C, h, w = shape
        torch.manual_seed(20 + C + cin)
        ref = to.AsppHeadOracle(cin, RATES, RATES, C)
        from rnd_semantic_segmentation_b200 import ASPP_Classifier_V2
        torch.manual_seed(20 + C + cin)
        ours = ASPP_Classifier_V2(cin, RATES, RATES, C).cuda()
        g = torch.Generator().manual_seed(21 + h + cin)
        x = torch.relu(torch.randn(n, cin, h, w, generator=g))
        go = torch.randn(n, C, h, w, generator=g) * 1e-4
        eff = effective_bf16_head(ref).double()
        xr = bf16_round(x).double().requires_grad_(True)
        want = eff(xr)
        want.backward(bf16_round(go).double())
        wgrads = []
        for m in eff.conv2d_list:
            wg = m.weight.grad.clone()
            wg[:, :, 1, 1] = eff.conv2d_list[0].weight.grad[:, :, 1, 1]      # d/dW_r(centre) is the same for every branch
            wgrads.append(wg)
        _ORACLE[shape] = (ours, x, go, want.detach(), xr.grad, wgrads)
    return _ORACLE[shape]


def _run(lib, shape, setting):
    ours, x, go, *_ = _head(shape)
    set_switches(lib, **dict(DEFAULT, **setting))
    try:
        ours.zero_grad(set_to_none=True)
        xc = x.cuda().requires_grad_(True)
        y = ours(xc)
        y.backward(go.cuda())
        torch.cuda.synchronize()
        return y.detach().clone(), xc.grad.clone(), [m.weight.grad.clone() for m in ours.conv2d_list]
    finally:
        set_switches(lib, **DEFAULT)


@pytest.mark.parametrize("setting", list(SETTINGS), ids=str)
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_head_under_switch(lib, shape, setting):
    _, _, go, want, want_gx, want_w = _head(shape)
    if shape not in _DEFAULT:
        _DEFAULT[shape] = _run(lib, shape, {})
    y0, gx0, w0 = _DEFAULT[shape]
    y, gx, w = _run(lib, shape, SETTINGS[setting])
    assert rel_err(y, want) <= TOL
    assert rel_err(gx, want_gx) <= TOL
    for i, (a, b) in enumerate(zip(w, want_w)):
        assert rel_err(a, b) <= TOL, f"branch {i}"
    assert torch.equal(y.view(torch.int32), y0.view(torch.int32)), rel_err(y, y0)
    assert torch.equal(gx.view(torch.int32), gx0.view(torch.int32)), rel_err(gx, gx0)
    for i, (a, b) in enumerate(zip(w, w0)):
        assert rel_err(a, b) <= WGRAD_REORDER, f"branch {i}: {rel_err(a, b)}"


@pytest.mark.parametrize("setting", ["default", "sharing0", "sharing5"])
@pytest.mark.parametrize("shape", [(1, 64, 256, 8, 16), (1, 512, 2048, 5, 7)], ids=str)
def test_seam_conv3_single_m_tile(lib, shape, setting):
    """P <= 128 pixels: one M-tile, so the seam GEMM drops its pair -- the SEAM kernel on one CTA."""
    import rnd_semantic_segmentation_b200 as b200
    N, Cin, Cout, h, w = shape
    out2, identity, W, scale, bias = _op_inputs(N, Cin, Cout, h, w, 17)
    set_switches(lib, **dict(DEFAULT, **SETTINGS[setting]))
    try:
        y = b200.seam_conv3_tail(out2, identity, W, scale, bias)
        torch.cuda.synchronize()
    finally:
        set_switches(lib, **DEFAULT)
    _check_against_oracle(y, out2, identity, W, scale, bias)
