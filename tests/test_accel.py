"""`zuko_b200.accelerate(flow)` — the drop-in seam of SURVEY §8(b): an engine-backed
LazyDistribution that shares the parameters / buffers of an existing flow.

CPU part: structure, sharing and error behaviour, against flows built by the constructors of the
*unmodified reference* (rebuilt from their recorded module trees, tests/golden/make_golden_accel.py)
and against the engine's own modules.  GPU part: the accelerated flow reproduces the golden
log-densities and follows in-place updates of the source flow.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

import zuko_b200
from zuko_b200.accel import _convert, _share

from cases import GOLDEN, SMALL_CASES, assert_log_prob_parity, build_flow, load
from module_tree import rebuild

REJECTED = ("maf_prelu", "naf", "gf", "maf_float64")  # options the engine does not implement


def _reference_flows():
    """Fresh copies of the reference-built flows: the reference's class names, constructor attributes,
    masks, orders and state-dict layout (tests/module_tree.py)."""
    with np.load(GOLDEN / "accel_reference_flows.npz") as payload:
        return rebuild(payload)


def _assert_shared(acc, src):
    sd_src, sd_acc = src.state_dict(), acc.state_dict()
    assert list(sd_src) == list(sd_acc)
    for k in sd_src:
        assert sd_src[k].data_ptr() == sd_acc[k].data_ptr() and sd_src[k].shape == sd_acc[k].shape, k
    p_src, p_acc = dict(src.named_parameters()), dict(acc.named_parameters())
    assert all(p_src[k] is p_acc[k] for k in p_src)
    b_src, b_acc = dict(src.named_buffers()), dict(acc.named_buffers())
    assert all(b_src[k] is b_acc[k] for k in b_src)


def test_accelerate_reference_flows_share_tensors():
    for name, src in _reference_flows().items():
        if name in REJECTED:
            continue
        acc = zuko_b200.accelerate(src)
        assert isinstance(acc, zuko_b200.lazy.LazyDistribution), name
        _assert_shared(acc, src)
        # every lazy layer was replaced by its engine counterpart
        for t in acc.transform.transforms:
            assert type(t).__module__.startswith("zuko_b200."), (name, type(t))


def test_accelerate_keeps_reference_built_masks_and_orders():
    src = _reference_flows()["maf_randperm"]
    acc = zuko_b200.accelerate(src)
    for ts, ta in zip(src.transform.transforms, acc.transform.transforms, strict=True):
        assert ta.passes == ts.passes and torch.equal(ta.order, ts.order)
        for ms, ma in zip(ts.hyper, ta.hyper, strict=True):
            if hasattr(ms, "mask"):
                assert ma.mask is ms.mask
    adj = zuko_b200.accelerate(_reference_flows()["adjacency"])
    assert adj.transform.transforms[0].order is None and adj.transform.transforms[0].passes == 3


def test_accelerate_sees_updates_of_the_source():
    src = _reference_flows()["nsf"]
    acc = zuko_b200.accelerate(src)
    layer = acc.transform.transforms[0]
    sig0 = layer._layer_signature()
    with torch.no_grad():
        src.transform.transforms[0].hyper[0].weight.mul_(1.5)  # an optimizer step on the reference module
    assert layer._layer_signature() != sig0  # -> the packed weights are rebuilt on the next call
    # load_state_dict on the source copies in place: still shared
    src.load_state_dict({k: torch.zeros_like(v) for k, v in src.state_dict().items()})
    assert float(acc.transform.transforms[1].hyper[2].weight.detach().abs().sum()) == 0.0
    # .to() / _apply replace buffer objects: detected and re-adopted at the next forward
    src._apply(lambda t: t.clone())
    assert acc._stale()
    acc.resync()
    _assert_shared(acc, src)


def test_accelerate_rejects_what_the_engine_does_not_implement():
    flows = _reference_flows()
    for bad in ("maf_prelu", "naf", "gf"):
        with pytest.raises(NotImplementedError, match="accelerate"):
            zuko_b200.accelerate(flows[bad])
    with pytest.raises(TypeError, match="float32"):
        zuko_b200.accelerate(flows["maf_float64"])
    with pytest.raises(TypeError, match="lazy Flow"):
        zuko_b200.accelerate(torch.nn.Linear(2, 2))


@pytest.mark.parametrize("name", SMALL_CASES)
def test_accelerate_engine_modules_by_name(name):
    """The converters recognise modules by class name / constructor attributes, so the engine's
    own modules (same names as the reference's) exercise them where the reference is absent."""
    src = build_flow(name)
    mirror = _convert(src, passthrough=False)
    assert mirror is not src and list(mirror.state_dict()) == list(src.state_dict())
    _share(mirror, src)
    _assert_shared(zuko_b200.accelerate(src), src)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL_CASES + ["cfg2_nsf"])
def test_accelerated_flow_matches_golden(device, name):
    g = load(f"flow_{name}")
    src = build_flow(name, g).to(device)
    if "w_scale" in g:
        for t in src.transform.transforms:
            if hasattr(t, "hyper"):
                t.hyper.gemm_mode = "fp32"
    acc = zuko_b200.accelerate(src)
    if "w_scale" in g:
        for t in acc.transform.transforms:
            if hasattr(t, "hyper"):
                t.hyper.gemm_mode = "fp32"
    x = torch.from_numpy(g["x"]).to(device)
    c = torch.from_numpy(g["c"]).to(device) if "c" in g and g["c"].size else None
    with torch.no_grad():
        lp = acc(c).log_prob(x)
        assert_log_prob_parity(lp.cpu().numpy(), g, rtol=1e-5)
        # an in-place update of the source is seen through the shared tensors
        first = next(p for p in src.parameters())
        first.mul_(1.25)
        assert torch.equal(acc(c).log_prob(x), src(c).log_prob(x))
        assert not torch.equal(acc(c).log_prob(x), lp)


@pytest.mark.gpu
def test_accelerate_after_move_to_device(device):
    """`accelerate` on the CPU module, then `.to(device)` on the SOURCE: the buffer objects are
    replaced by torch; the accelerated flow re-adopts them at the next call."""
    g = load("flow_nsf35_row")
    src = build_flow("nsf35_row", g)
    acc = zuko_b200.accelerate(src)
    src.to(device)
    x = torch.from_numpy(g["x"]).to(device)
    c = torch.from_numpy(g["c"]).to(device)
    with torch.no_grad():
        assert_log_prob_parity(acc(c).log_prob(x).cpu().numpy(), g, rtol=1e-5)


def test_accelerate_leaves_the_global_rng_alone():
    """The mirror's constructors draw initial weights that are thrown away: the caller's RNG stream must
    not move (ADVICE r1)."""
    torch.manual_seed(123)
    flow = zuko_b200.flows.NSF(3, 2, transforms=2, hidden_features=[16])
    torch.manual_seed(7)
    a = torch.rand(3)
    torch.manual_seed(7)
    zuko_b200.accelerate(flow)
    b = torch.rand(3)
    assert torch.equal(a, b)
