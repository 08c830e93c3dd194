"""Parity of the CUDA path (through the C ABI) with the reference's golden outputs and with the CPU oracle.

Tolerance: 1e-5 relative (`rel_err`: max |a-b| / max(|a|,|b|,1)), the bar BASELINE.json states for fp32;
identity columns and permutations must be bit-exact.  Per-layer log|det| of a spline layer additionally gets
the fp64 sandwich of SURVEY.md section 8c where the reference's own fp32 round-off exceeds 1e-5."""
import pytest
import torch

from conftest import load_golden, rel_err
from nflows_b200 import _native
from nflows_b200 import config
from nflows_b200 import kernels as K
from nflows_b200 import transforms as T
from nflows_b200.flows import recipes
from nflows_b200.nn.nets import MLP, ResidualNet
from nflows_b200.transforms.splines import rational_quadratic as rq
from nflows_b200.utils import torchutils
from oracle import flow_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5


class native_launches:
    """Asserts that the block launched our kernels (no silent torch fallback)."""

    def __enter__(self):
        self.before = _native.launch_count()
        return self

    def __exit__(self, *exc):
        if exc[0] is None:
            assert _native.launch_count() > self.before, "no native kernel was launched"


def to_dev(module, dev):
    return module.eval().to(dev)


@torch.no_grad()
def test_searchsorted_and_identity_spline(cuda_device):
    # identity-init known answer (reference tests/transforms/splines/rational_quadratic_test.py:33-62, 116-146)
    shape, k = (2, 3, 4), 10
    zeros = torch.zeros(*shape, k, device=cuda_device)
    x = torch.rand(*shape, device=cuda_device)
    with native_launches():
        y, lad = rq.rational_quadratic_spline(x, zeros, zeros, torch.zeros(*shape, k + 1, device=cuda_device),
                                              enable_identity_init=True)
    assert rel_err(y.cpu(), x.cpu()) <= 1e-6 and float(lad.abs().max()) <= 1e-6
    # linear tails: identity outside [-B, B] and in the interior bins; the two edge bins are NOT the identity
    # because the boundary-derivative constant ignores beta (reference rational_quadratic.py:33-36 vs :100-104)
    xt = (torch.rand(*shape, device=cuda_device) - 0.5) * 4
    zd = torch.zeros(*shape, k - 1, device=cuda_device)
    y, lad = rq.unconstrained_rational_quadratic_spline(xt, zeros, zeros, zd, enable_identity_init=True)
    interior = (xt.abs() < 0.8) | (xt.abs() > 1.0)
    assert rel_err(y[interior].cpu(), xt[interior].cpu()) <= 1e-6 and float(lad[interior].abs().max()) <= 1e-6
    wy, wl = O.rq_spline_unconstrained(xt.cpu(), zeros.cpu(), zeros.cpu(), zd.cpu(), enable_identity_init=True)
    assert rel_err(y.cpu(), wy) <= TOL and rel_err(lad.cpu(), wl) <= TOL


def _elementwise_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    both_nan = torch.isnan(a) & torch.isnan(b)
    err = (a - b).abs() / torch.maximum(torch.maximum(a.abs(), b.abs()), torch.ones_like(a))
    return torch.where(both_nan, torch.zeros_like(err), err).flatten().sort().values


def assert_statistically_as_accurate(got, ref32, truth, what):
    """Stress vectors with deliberately sharp bins are ill-conditioned next to knots (a 1-ulp knot difference moves
    theta by percents), so ANY fp32 evaluation has a heavy error tail there and the single worst element is luck.
    Criterion: the error distribution against the fp64 truth must match the reference's: 99th / 99.9th percentile
    within 2x (+1e-5), worst element within 15x of the reference's worst (profiles/parity_calibration_r2.txt, captured with
    the shipped kernels: the largest observed ratio is 10.1, on the log|det| of the sharpest constrained-spline vectors)."""
    e, r = _elementwise_err(got, truth), _elementwise_err(ref32, truth)
    n = len(e)
    for q in (0.99, 0.999):
        i = min(n - 1, int(q * n))
        assert e[i] <= 2 * r[i] + TOL, (what, q, float(e[i]), float(r[i]))
    assert e[-1] <= 15 * r[-1] + TOL, (what, "max", float(e[-1]), float(r[-1]))


@torch.no_grad()
def test_spline_function_vectors(cuda_device):
    g = load_golden("spline")
    dev = lambda k: g[k].to(cuda_device)
    box = dict(left=-1.0, right=3.0, bottom=-1.0, top=3.0, min_bin_width=1e-2, min_bin_height=2e-2, min_derivative=5e-2)
    for inv in (False, True):
        with native_launches():
            y, l = rq.unconstrained_rational_quadratic_spline(dev("x_tails"), dev("uw"), dev("uh"), dev("ud_tails"), inverse=inv,
                                                              tails="linear", tail_bound=g["tail_bound"])
        wy, wl = g["tails_inv%d" % inv]
        ty, tl = O.rq_spline_unconstrained(g["x_tails"].double(), g["uw"].double(), g["uh"].double(), g["ud_tails"].double(),
                                           inverse=inv, tail_bound=g["tail_bound"])
        assert_statistically_as_accurate(y, wy, ty, ("tails y", inv))
        assert_statistically_as_accurate(l, wl, tl, ("tails lad", inv))
        # exact edge semantics (SURVEY Appendix A): x=-B -> (-B, ~0); outside -> identity, lad 0; NaN -> NaN, lad 0
        assert float(y[0]) == -3.0 and abs(float(l[0])) <= 2e-7
        assert float(y[2]) == float(g["x_tails"][2]) and float(l[2]) == 0.0
        assert torch.isnan(y[6]) and float(l[6]) == 0.0 and float(y[7]) == float(g["x_tails"][7])
        for key, xin, kw in (("constrained_inv%d", g["x_constrained"], {}), ("constrained_box_inv%d", g["x_constrained"] * 4 - 1, box)):
            y, l = rq.rational_quadratic_spline(xin.to(cuda_device), dev("uw"), dev("uh"), dev("ud_constrained"), inverse=inv, **kw)
            wy, wl = g[key % inv]
            ty, tl = O.rq_spline(xin.double(), g["uw"].double(), g["uh"].double(), g["ud_constrained"].double(), inverse=inv, **kw)
            assert_statistically_as_accurate(y, wy, ty, (key, "y", inv))
            assert_statistically_as_accurate(l, wl, tl, (key, "lad", inv))


@torch.no_grad()
def test_spline_error_conventions(cuda_device):
    k = 4
    z = torch.zeros(5, k, device=cuda_device)
    d = torch.zeros(5, k + 1, device=cuda_device)
    x = torch.tensor([0.1, 0.5, 1.5, 0.2, 0.3], device=cuda_device)
    with pytest.raises(T.InputOutsideDomain):
        rq.rational_quadratic_spline(x, z, z, d)
    with pytest.raises(ValueError):
        rq.rational_quadratic_spline(x.clamp(0, 1), z, z, d, min_bin_width=0.3)
    with pytest.raises(RuntimeError):
        rq.unconstrained_rational_quadratic_spline(x, z, z, d[:, :k - 1], tails="cubic")
    # empty input is fine
    e = torch.zeros(0, device=cuda_device)
    y, l = rq.rational_quadratic_spline(e, z[:0], z[:0], d[:0])
    assert y.shape == (0,) and l.shape == (0,)


@torch.no_grad()
def test_cfg1_affine_flow(cuda_device):
    g = load_golden("cfg1_affine")
    flow = recipes.affine_flow_2d()
    flow.load_state_dict(g["sd"])
    flow = to_dev(flow, cuda_device)
    x = g["x"].to(cuda_device)
    with native_launches():
        lp = flow.log_prob(x)
    assert rel_err(lp.cpu(), g["log_prob"]) <= TOL
    z, lad = flow._transform(x)
    assert rel_err(z.cpu(), g["z"]) <= TOL and rel_err(lad.cpu(), g["lad"]) <= TOL
    xr, ladr = flow._transform.inverse(g["z"].to(cuda_device))
    assert rel_err(xr.cpu(), g["x_roundtrip"]) <= TOL and rel_err(ladr.cpu(), g["lad_inverse"]) <= TOL
    # identity halves are bit-exact (reference tests/transforms/coupling_test.py:50)
    t0 = flow._transform._transforms[0]
    y0, _ = t0(x)
    assert torch.equal(y0[:, t0.identity_features], x[:, t0.identity_features])
    assert flow.sample(5).shape == (5, 2)
    s, lps = flow.sample_and_log_prob(64)
    assert rel_err(lps.cpu(), flow.log_prob(s).cpu()) <= 1e-4


@torch.no_grad()
def test_affine_variants(cuda_device):
    g = load_golden("affine_variants")
    f = lambda i, o: ResidualNet(i, o, hidden_features=16)
    mask = torchutils.create_mid_split_binary_mask(10)
    tg = T.AffineCouplingTransform(mask, f, scale_activation=T.AffineCouplingTransform.GENERAL_SCALE_ACTIVATION)
    tg.load_state_dict(g["sd_general"])
    tg = to_dev(tg, cuda_device)
    x = g["x"].to(cuda_device)
    with native_launches():
        y, l = tg(x)
    assert rel_err(y.cpu(), g["y_general"]) <= TOL and rel_err(l.cpu(), g["lad_general"]) <= TOL
    y, l = tg.inverse(x)
    assert rel_err(y.cpu(), g["xinv_general"]) <= TOL and rel_err(l.cpu(), g["ladinv_general"]) <= TOL
    ta = T.AdditiveCouplingTransform(mask, f)
    ta.load_state_dict(g["sd_additive"])
    ta = to_dev(ta, cuda_device)
    with native_launches():
        y, l = ta(x)
    assert rel_err(y.cpu(), g["y_additive"]) <= TOL and torch.equal(l.cpu(), torch.zeros(x.shape[0]))


@torch.no_grad()
def test_cfg2_rq_coupling(cuda_device):
    g = load_golden("cfg2_rq_coupling")
    t = recipes.rq_coupling_layer()
    t.load_state_dict(g["sd"])
    t = to_dev(t, cuda_device)
    x = g["x"].to(cuda_device)
    for suffix in ("", "_x3"):
        if suffix:
            for name, p in t.named_parameters():
                if "final_layer" in name:
                    p.mul_(3.0)
        with native_launches():
            y, l = t(x)
        assert rel_err(y.cpu(), g["y" + suffix]) <= TOL and rel_err(l.cpu(), g["lad" + suffix]) <= 3e-5
        assert torch.equal(y[:, t.identity_features], x[:, t.identity_features])
        xi, li = t.inverse(x)
        assert rel_err(xi.cpu(), g["xinv" + suffix]) <= (TOL if not suffix else 1e-4)
        assert rel_err(li.cpu(), g["ladinv" + suffix]) <= (3e-5 if not suffix else 1e-3)
        back, lb = t.inverse(y)
        assert rel_err(back.cpu(), g["x"]) <= 1e-4


@torch.no_grad()
def test_rq_coupling_constrained_and_domain_error(cuda_device):
    g = load_golden("rq_coupling_constrained")
    t = T.PiecewiseRationalQuadraticCouplingTransform(
        mask=torchutils.create_mid_split_binary_mask(11),
        transform_net_create_fn=lambda i, o: ResidualNet(i, o, hidden_features=24, num_blocks=1),
        num_bins=5, tails=None, min_bin_width=2e-3, min_bin_height=3e-3, min_derivative=4e-3)
    t.load_state_dict(g["sd"])
    t = to_dev(t, cuda_device)
    x = g["x"].to(cuda_device)
    with native_launches():
        y, l = t(x)
    assert rel_err(y.cpu(), g["y"]) <= TOL and rel_err(l.cpu(), g["lad"]) <= 3e-5
    xi, li = t.inverse(x)
    assert rel_err(xi.cpu(), g["xinv"]) <= 1e-4 and rel_err(li.cpu(), g["ladinv"]) <= 1e-3
    with pytest.raises(T.InputOutsideDomain):
        t(x + 1.0)
    with pytest.raises(ValueError):
        t(x[:, :5])


@torch.no_grad()
def test_unrecognised_conditioner_uses_spline_epilogue_kernel(cuda_device):
    """A conditioner that is not a relu ResidualNet/MLP runs in torch; the spline epilogue is still ours."""

    class Odd(torch.nn.Module):
        def __init__(self, i, o):
            super().__init__()
            self.hidden_features = 16
            self.a, self.b = torch.nn.Linear(i, 16), torch.nn.Linear(16, o)

        def forward(self, x, context=None):
            return self.b(torch.tanh(self.a(x)))

    torch.manual_seed(0)
    t = T.PiecewiseRationalQuadraticCouplingTransform(torchutils.create_alternating_binary_mask(9), Odd, num_bins=6,
                                                      tails="linear", tail_bound=2.0).eval()
    x = torch.randn(333, 9)
    sd = {k: v.clone() for k, v in t.state_dict().items()}
    idf, trf = sd["identity_features"], sd["transform_features"]
    params = t.transform_net(x[:, idf]).reshape(333, len(trf), -1)
    yt, lad = O.rq_spline_unconstrained(x[:, trf], params[..., :6] / 4.0, params[..., 6:12] / 4.0, params[..., 12:].clone(),
                                        tail_bound=2.0)
    t = t.to(cuda_device)
    with native_launches():
        y, l = t(x.to(cuda_device))
    assert rel_err(y[:, trf.to(cuda_device)].cpu(), yt) <= TOL and rel_err(l.cpu(), lad.sum(1)) <= 3e-5
    # MLP conditioner goes through the dense chain
    t2 = T.PiecewiseRationalQuadraticCouplingTransform(
        torchutils.create_alternating_binary_mask(9), lambda i, o: MLP([i], [o], [32, 32]), num_bins=6, tails="linear",
        tail_bound=2.0).eval()
    with pytest.warns(UserWarning):
        y_cpu, l_cpu = t2(x)
    t2 = t2.to(cuda_device)
    with pytest.warns(UserWarning):
        y2, l2 = t2(x.to(cuda_device))
    assert rel_err(y2.cpu(), y_cpu) <= TOL and rel_err(l2.cpu(), l_cpu) <= 3e-5


@torch.no_grad()
def test_linear_transforms(cuda_device):
    g = load_golden("linear_transforms")
    d = g["x"].shape[1]
    an, lu, pm = T.ActNorm(d), T.LULinear(d, identity_init=False), T.RandomPermutation(d)
    an.load_state_dict(g["sd_actnorm"]); lu.load_state_dict(g["sd_lu"]); pm.load_state_dict(g["sd_perm"])
    x = g["x"].to(cuda_device)
    for name, m in (("actnorm", an), ("lu", lu), ("perm", pm)):
        m = to_dev(m, cuda_device)
        with native_launches():
            y, l = m(x)
        assert rel_err(y.cpu(), g[name + "_y"]) <= TOL and rel_err(l.cpu(), g[name + "_lad"]) <= TOL, name
        y, l = m.inverse(x)
        assert rel_err(y.cpu(), g[name + "_xinv"]) <= 1e-4 and rel_err(l.cpu(), g[name + "_ladinv"]) <= TOL, name
    y, _ = pm(x)
    assert torch.equal(y.cpu(), g["x"][:, g["sd_perm"]["_permutation"]])        # bit-exact indexing
    y, _ = pm.inverse(y)
    assert torch.equal(y, x)
    # parameter update invalidates the folded-weight cache
    lu.bias.add_(1.0)
    y2, _ = lu(x)
    assert rel_err(y2.cpu(), g["lu_y"] + 1.0) <= TOL


@torch.no_grad()
def test_nsf_small_flow_fused_and_unfused(cuda_device):
    g = load_golden("nsf_small")
    flow = recipes.rq_nsf(g["features"], g["hidden"], g["layers"])
    flow.load_state_dict(g["sd"])
    flow = to_dev(flow, cuda_device)
    x = g["x"].to(cuda_device)
    with native_launches():
        lp = flow.log_prob(x)
    assert rel_err(lp.cpu(), g["log_prob"]) <= TOL
    z, lad = flow._transform(x)
    assert rel_err(z.cpu(), g["z"]) <= 5e-5 and rel_err(lad.cpu(), g["lad"]) <= 5e-5
    xs, lads = flow._transform.inverse(g["noise"].to(cuda_device))
    # the inverse amplifies rounding noise ~1000x (the reference's own fp32 result is 6e-5 from the fp64 value), so it is
    # judged against the fp64 result of the same module's torch path (pinned to the reference in test_api_eager_golden.py)
    # with the reference's fp32 distance as the yardstick
    f64 = recipes.rq_nsf(g["features"], g["hidden"], g["layers"])
    f64.load_state_dict(g["sd"])
    xs64, lads64 = f64.double().eval()._transform.inverse(g["noise"].double())
    assert rel_err(xs.cpu(), xs64) <= max(1e-5, 4 * rel_err(g["sample"], xs64))
    assert rel_err(lads.cpu(), lads64) <= max(1e-5, 4 * rel_err(g["lad_inverse"], lads64))
    # transform-by-transform (no affine folding) agrees with the folded chain
    out, total = x, torch.zeros(x.shape[0], device=cuda_device)
    for t in flow._transform._transforms:
        out, l = t(out)
        total += l
    assert rel_err(out, z) <= 5e-5 and rel_err(total, lad) <= 5e-5
    # ragged / tiny batches
    for n in (1, 3, 130):
        assert rel_err(flow.log_prob(x[:n]).cpu(), g["log_prob"][:n]) <= TOL
    assert flow.log_prob(x[:0]).shape == (0,)


@torch.no_grad()
def test_nsf784_layer_and_full_flow_seeded(cuda_device):
    """Full-shape cfg-3 weights re-created from the seed (the fixture stores only inputs/outputs/checksum)."""
    for name in ("nsf784_layer", "nsf784_full"):
        g = load_golden(name)
        torch.manual_seed(g["seed"])
        flow = recipes.perturb_(recipes.rq_nsf(g["features"], g["hidden"], g["layers"]).eval(), g["perturb_seed"])
        ck = float(sum(v.double().abs().sum() for v in flow.state_dict().values() if v.is_floating_point()))
        if abs(ck - g["checksum"]) > 1e-9 * abs(g["checksum"]):
            pytest.fail("weights re-created from the seed do not match the fixture's checksum (torch CPU RNG stream changed?): "
                        "regenerate tests/golden with oracle/make_golden.py against the reference")
        flow = to_dev(flow, cuda_device)
        x = g["x"].to(cuda_device)
        with native_launches():
            lp = flow.log_prob(x)
        assert rel_err(lp.cpu(), g["log_prob"]) <= TOL, name
        if name == "nsf784_layer":
            z, lad = flow._transform(x)
            assert rel_err(z.cpu(), g["z"]) <= TOL
            # fp64 sandwich for the per-layer log|det| (the reference itself is ~3e-5 from fp64 here)
            ref_gap = rel_err(g["lad"], g["lad_fp64"])
            assert rel_err(lad.cpu(), g["lad_fp64"]) <= max(3 * ref_gap, TOL)
            xi, li = flow._transform.inverse(x)
            assert rel_err(xi.cpu(), g["xinv"]) <= 1e-4 and rel_err(li.cpu(), g["ladinv"]) <= 1e-4
        else:
            assert rel_err(lp.cpu(), g["log_prob_fp64"]) <= TOL


@torch.no_grad()
def test_cfg3_full_shape_many_tiles_rounds_and_clusters(cuda_device):
    """BASELINE configs[2] at its full shape (D=784, H=256, 10 layers) on a batch that spans many 128-row tiles, several
    clusters per SM and several launch rounds (blocks forced to 2^13 rows), with a ragged tail: 1024 random rows against the CPU
    oracle at 1e-5, and bit-for-bit agreement with other block sizes / batch splits (rows are independent)."""
    torch.manual_seed(0)
    flow = recipes.perturb_(recipes.rq_nsf(784, 256, 10).eval())
    sd = {k: v.clone() for k, v in flow.state_dict().items()}
    flow = flow.to(cuda_device)
    gen = torch.Generator(device=cuda_device).manual_seed(21)
    n = (1 << 15) + 77
    x = torch.randn(n, 784, device=cuda_device, generator=gen)
    saved = (config.trunk_block_rows, config.affine_block_rows, config.coupling_block_rows)
    config.trunk_block_rows = config.affine_block_rows = config.coupling_block_rows = 1 << 13
    try:
        with native_launches():
            lp = flow.log_prob(x)
    finally:
        config.trunk_block_rows, config.affine_block_rows, config.coupling_block_rows = saved
    assert bool(torch.isfinite(lp).all())
    assert torch.equal(lp, flow.log_prob(x))                                                  # default 2^19-row blocks
    assert torch.equal(lp, torch.cat([flow.log_prob(x[:10001]), flow.log_prob(x[10001:])]))   # another split, other tile phases
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(3))[:1024]
    want = O.flow_log_prob(sd, O.nsf_spec(10), x[idx.to(cuda_device)].cpu())
    assert rel_err(lp[idx.to(cuda_device)].cpu(), want) <= TOL


@torch.no_grad()
def test_oracle_parity_on_random_rows_of_a_large_batch(cuda_device):
    """Rows are independent: run a large batch on the GPU, check a random subset against the CPU oracle."""
    torch.manual_seed(0)
    flow = recipes.perturb_(recipes.rq_nsf(features=96, hidden_features=64, num_layers=4).eval())
    sd = {k: v.clone() for k, v in flow.state_dict().items()}
    flow = flow.to(cuda_device)
    gen = torch.Generator(device=cuda_device).manual_seed(5)
    x = torch.randn(1 << 17, 96, device=cuda_device, generator=gen) * 1.5
    lp = flow.log_prob(x)
    rows = torch.randint(0, x.shape[0], (2048,), generator=torch.Generator().manual_seed(6))
    want = O.flow_log_prob(sd, O.nsf_spec(4), x[rows.to(cuda_device)].cpu())
    assert rel_err(lp[rows.to(cuda_device)].cpu(), want) <= TOL
    # chunk-consistency: a different batch split gives the same per-row numbers bit-for-bit
    assert torch.equal(flow.log_prob(x[: 1 << 12]), lp[: 1 << 12])
    # encode -> decode round trip at scale
    z = flow.transform_to_noise(x[: 1 << 14])
    back, _ = flow._transform.inverse(z)
    assert rel_err(back, x[: 1 << 14]) <= 2e-3


@torch.no_grad()
def test_domain_check_can_be_disabled(cuda_device):
    k = 4
    z = torch.zeros(3, k, device=cuda_device)
    d = torch.zeros(3, k + 1, device=cuda_device)
    x = torch.tensor([0.1, 1.5, 0.3], device=cuda_device)
    config.check_domain = False
    try:
        y, _ = rq.rational_quadratic_spline(x, z, z, d)
        assert y.shape == (3,)
    finally:
        config.check_domain = True


@torch.no_grad()
@pytest.mark.parametrize("bins,tails", [(8, "linear"), (10, "linear"), (4, "linear"), (16, "linear"), (8, None), (10, None),
                                       (16, None)])
def test_fused_coupling_kernel_matches_unfused_and_oracle(cuda_device, bins, tails, monkeypatch):
    """The one-kernel final-layer+spline path against (a) the GEMM -> HBM params -> spline-kernel path with the FFMA GEMM
    and (b) the CPU oracle, forward and inverse, ragged row count, odd feature count."""
    torch.manual_seed(bins)
    d = 48   # 24 identity features (a multiple of 4, as the TMA path needs), 24 transformed
    t = T.PiecewiseRationalQuadraticCouplingTransform(
        torchutils.create_alternating_binary_mask(d), lambda i, o: ResidualNet(i, o, hidden_features=64, num_blocks=1),
        num_bins=bins, tails=tails, tail_bound=2.5).eval()
    for name, p in t.named_parameters():
        if "final_layer" in name:
            p.mul_(2.0)
    x = torch.rand(700, d) if tails is None else torch.randn(700, d) * 1.3
    sd = {k: v.clone() for k, v in t.state_dict().items()}
    kw = dict(num_bins=bins, tails=tails, tail_bound=2.5)
    t = t.to(cuda_device)
    xd = x.to(cuda_device)
    for inverse in (False, True):
        want_y, want_l = O.rq_coupling({k: v.clone() for k, v in sd.items()}, "", x, inverse=inverse, **kw)
        truth_y, truth_l = O.rq_coupling({k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}, "",
                                         x.double(), inverse=inverse, **kw)
        run = (lambda: t.inverse(xd)) if inverse else (lambda: t(xd))
        config.fuse_coupling = True
        before = _native.launch_count()
        y1, l1 = run()
        fused_launches = _native.launch_count() - before
        config.fuse_coupling = False
        monkeypatch.setenv("NFLOWS_B200_GEMM", "simt")
        try:
            before = _native.launch_count()
            y2, l2 = run()
            unfused_launches = _native.launch_count() - before
        finally:
            config.fuse_coupling = True
            monkeypatch.delenv("NFLOWS_B200_GEMM")
        tol_y = max(TOL, 3 * rel_err(want_y, truth_y))
        tol_l = max(3e-5, 5 * rel_err(want_l, truth_l))
        assert rel_err(y1.cpu(), truth_y) <= tol_y and rel_err(y2.cpu(), truth_y) <= tol_y, (bins, tails, inverse)
        assert rel_err(l1.cpu(), truth_l) <= tol_l and rel_err(l2.cpu(), truth_l) <= tol_l, (bins, tails, inverse)
        idf = sd["identity_features"].to(cuda_device)
        assert torch.equal(y1[:, idf], xd[:, idf]) and torch.equal(y2[:, idf], xd[:, idf])


@torch.no_grad()
def test_next_rows_against_reference_goldens(cuda_device):
    """SURVEY section 8 'next' rows that run on our kernels, against outputs of the UNMODIFIED reference (tests/golden/next_rows.pt,
    oracle/make_golden.py next_rows): 1x1 convolution on image batches (folded LU dense layer per pixel), unconditional RQ CDF
    (batch-shared spline parameters, both tail modes), an RQ coupling with apply_unconditional_transform, SimpleRealNVP, and an
    MLP-conditioned RQ coupling.  Weights are the reference's state_dicts."""
    from nflows_b200.flows import SimpleRealNVP
    g = load_golden("next_rows")

    for key, channels in (("conv1x1", 3), ("conv1x1_c12", 12)):
        r = g[key]
        conv = T.OneByOneConvolution(channels, identity_init=False).eval()
        conv.load_state_dict(r["sd"], strict=True)
        conv = conv.to(cuda_device)
        with native_launches():
            got, gl = conv(r["x"].to(cuda_device))
        assert rel_err(got.cpu(), r["y"]) <= TOL and rel_err(gl.cpu(), r["lad"]) <= TOL, key
        if "xinv" in r:
            back, bl = conv.inverse(r["x"].to(cuda_device))
            assert rel_err(back.cpu(), r["xinv"]) <= 1e-4 and rel_err(bl.cpu(), r["ladinv"]) <= TOL, key

    for tails in (None, "linear"):
        r = g["rq_cdf_%s" % (tails or "none")]
        cdf = T.PiecewiseRationalQuadraticCDF(shape=[7], num_bins=6, tails=tails, tail_bound=2.0).eval()
        cdf.load_state_dict(r["sd"], strict=True)
        cdf = cdf.to(cuda_device)
        with native_launches():
            got, gl = cdf(r["x"].to(cuda_device))
        # randn * 1.5 logits without the 1/sqrt(H) scaling give sharp bins: the reference's own fp32 log|det| is ~1e-4 from an fp64
        # evaluation of the same parameters here, so the log|det| check is the fp64 sandwich (oracle in float64)
        n = r["x"].shape[0]
        ex = lambda t: t[None].expand(n, *t.shape).double()
        sd = r["sd"]
        spline = O.rq_spline_unconstrained if tails else O.rq_spline
        kw = dict(tail_bound=2.0) if tails else {}
        _, l64 = spline(r["x"].double(), ex(sd["unnormalized_widths"]), ex(sd["unnormalized_heights"]),
                        ex(sd["unnormalized_derivatives"]), inverse=False, **kw)
        l64 = l64.sum(dim=1)
        assert rel_err(got.cpu(), r["y"]) <= TOL, tails
        assert rel_err(gl.cpu(), l64) <= max(3e-5, 3 * rel_err(r["lad"], l64)), tails
        # the inverse on these sharp bins amplifies round-off: the reference's own fp32 inverse is 4e-4 .. 5e-4 from fp64 -> sandwich
        back, bl = cdf.inverse(r["inv_in"].to(cuda_device))
        x64, li64 = spline(r["inv_in"].double(), ex(sd["unnormalized_widths"]), ex(sd["unnormalized_heights"]),
                           ex(sd["unnormalized_derivatives"]), inverse=True, **kw)
        li64 = li64.sum(dim=1)
        assert rel_err(back.cpu(), x64) <= max(1e-4, 3 * rel_err(r["xinv"], x64)), tails
        assert rel_err(bl.cpu(), li64) <= max(1e-4, 3 * rel_err(r["ladinv"], li64)), tails

    r = g["rq_coupling_unconditional"]
    t = T.PiecewiseRationalQuadraticCouplingTransform(
        torchutils.create_alternating_binary_mask(16), lambda i, o: ResidualNet(i, o, hidden_features=32, num_blocks=1),
        num_bins=8, tails="linear", tail_bound=3.0, apply_unconditional_transform=True).eval()
    t.load_state_dict(r["sd"], strict=True)
    t = t.to(cuda_device)
    with native_launches():
        got, gl = t(r["x"].to(cuda_device))
    assert rel_err(got.cpu(), r["y"]) <= TOL and rel_err(gl.cpu(), r["lad"]) <= 3e-5
    gi, gil = t.inverse(r["x"].to(cuda_device))
    # the inverse amplifies round-off: sandwich against a float64 evaluation of the same module (CPU, torch path)
    import copy
    xi64, li64 = copy.deepcopy(t).cpu().double().inverse(r["x"].double())
    assert rel_err(gi.cpu(), xi64) <= max(1e-4, 3 * rel_err(r["xinv"], xi64))
    # log|det| of the INVERSE on sharpened bins (final layer x3 + noise, CDF logits x3): the quadratic root loses digits next to
    # knots; SURVEY Appendix C puts the reference's own fp32-vs-fp64 gap for this quantity at 4e-5 (x1) .. 4e-3 (x10)
    assert rel_err(gil.cpu(), li64) <= max(3e-4, 3 * rel_err(r["ladinv"], li64))

    r = g["simple_realnvp"]
    flow = SimpleRealNVP(features=10, hidden_features=16, num_layers=3, num_blocks_per_layer=2).eval()
    flow.load_state_dict(r["sd"], strict=True)
    with native_launches():
        got = flow.to(cuda_device).log_prob(r["x"].to(cuda_device))
    assert rel_err(got.cpu(), r["log_prob"]) <= TOL
    assert flow.sample(9).shape == (9, 10)

    # MLP conditioner: the reference's MLP takes no context argument, so the fixture was made with the usual user-side adapter
    # (transform_net.mlp.*); this package's MLP accepts the argument itself and is recognised as a dense chain
    r = g["rq_coupling_mlp"]
    t = T.PiecewiseRationalQuadraticCouplingTransform(
        torchutils.create_alternating_binary_mask(32), lambda i, o: MLP([i], [o], [64, 64, 64]),
        num_bins=8, tails="linear", tail_bound=3.0).eval()
    t.load_state_dict({k.replace("transform_net.mlp.", "transform_net."): v for k, v in r["sd"].items()}, strict=True)
    t = t.to(cuda_device)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # "Inputs to the softmax are not scaled down" (the reference warns as well)
        with native_launches():
            got, gl = t(r["x"].to(cuda_device))
        gi, gil = t.inverse(r["x"].to(cuda_device))
    assert rel_err(got.cpu(), r["y_fp64"]) <= max(TOL, 3 * rel_err(r["y"], r["y_fp64"]))
    assert rel_err(gl.cpu(), r["lad_fp64"]) <= max(3e-5, 3 * rel_err(r["lad"], r["lad_fp64"]))
    assert rel_err(gi.cpu(), r["xinv"]) <= 1e-4 and rel_err(gil.cpu(), r["ladinv"]) <= 1e-4


@torch.no_grad()
def test_context_conditioned_flow_against_reference_golden(cuda_device):
    """SURVEY section 8 row f4: Flow with an embedding net and context-conditioned ResidualNet conditioners (GLU gates) -- reference
    outputs in tests/golden/context_rows.pt.  Everything below the embedding net runs on our kernels: the folded affine runs,
    the gated conditioner (dense.Chain: context projection added to the initial layer, nfk_glu_skip_rows behind every block)
    and the fused final layer + spline."""
    from nflows_b200.distributions.normal import StandardNormal
    from nflows_b200.flows import Flow
    g = load_golden("context_rows")["context_flow"]
    features, ctx_raw, ctx = 16, 5, 6
    steps = []
    for i in range(3):
        steps.append(T.ActNorm(features))
        steps.append(T.CompositeTransform([T.RandomPermutation(features), T.LULinear(features, identity_init=True)]))
        steps.append(T.PiecewiseRationalQuadraticCouplingTransform(
            mask=torchutils.create_alternating_binary_mask(features, even=(i % 2 == 0)),
            transform_net_create_fn=lambda i_, o_: ResidualNet(i_, o_, hidden_features=32, context_features=ctx, num_blocks=2),
            num_bins=8, tails="linear", tail_bound=3.0))
    flow = Flow(T.CompositeTransform(steps), StandardNormal([features]), embedding_net=torch.nn.Linear(ctx_raw, ctx)).eval()
    flow.load_state_dict(g["sd"], strict=True)
    flow = flow.to(cuda_device)
    x, c = g["x"].to(cuda_device), g["context"].to(cuda_device)
    K.TIMELINE = []
    try:
        with native_launches():
            lp = flow.log_prob(x, context=c)
        tags = {t[0] for t in K.TIMELINE}
    finally:
        K.TIMELINE = None
    assert any(t.startswith("glu_skip_") for t in tags) and "rq_coupling_final" in tags, tags     # the gated conditioner ran natively
    assert rel_err(lp.cpu(), g["log_prob_fp64"]) <= max(TOL, 3 * rel_err(g["log_prob"], g["log_prob_fp64"]))
    assert rel_err(flow.transform_to_noise(x, context=c).cpu(), g["z"]) <= 5e-5
    # FFMA dense layers (NFLOWS_B200_GEMM=simt route of the same chain) agree
    import os
    os.environ["NFLOWS_B200_GEMM"] = "simt"
    try:
        assert rel_err(flow.log_prob(x, context=c).cpu(), g["log_prob_fp64"]) <= max(TOL, 3 * rel_err(g["log_prob"], g["log_prob_fp64"]))
    finally:
        os.environ.pop("NFLOWS_B200_GEMM")
    xs, _ = flow._transform.inverse(g["noise"].to(cuda_device), context=flow._embedding_net(c))
    assert rel_err(xs.cpu(), g["sample"]) <= 1e-3          # 3 spline inverses in a row: the reference's own round trip is ~1e-3
    assert flow.sample(4, context=c[:5]).shape == (5, 4, features)


@torch.no_grad()
def test_autoregressive_rq_transform_cfg4(cuda_device):
    """BASELINE configs[3]: MaskedPiecewiseRationalQuadraticAutoregressiveTransform D=64 K=8 -- forward (one MADE pass on the
    tensor-core dense chain + fused spline kernel) and the 64-pass inverse, against the reference's outputs."""
    g = load_golden("ar_rq")
    torch.manual_seed(g["seed"])
    ar = T.MaskedPiecewiseRationalQuadraticAutoregressiveTransform(features=64, hidden_features=256, num_bins=8, tails="linear",
                                                                   tail_bound=3.0, num_blocks=2).eval()
    for name, p in ar.named_parameters():
        if "final_layer" in name:
            p.mul_(g["final_scale"])
    ck = float(sum(v.double().abs().sum() for v in ar.state_dict().values() if v.is_floating_point()))
    if abs(ck - g["checksum"]) > 1e-9 * abs(g["checksum"]):
        pytest.fail("weights re-created from the seed do not match the fixture's checksum (torch CPU RNG stream changed?): "
                    "regenerate tests/golden with oracle/make_golden.py against the reference")
    ar = ar.to(cuda_device)
    x = g["x"].to(cuda_device)
    with native_launches():
        y, lad = ar(x)
    assert rel_err(y.cpu(), g["y_fp64"]) <= max(TOL, 3 * rel_err(g["y"], g["y_fp64"]))
    assert rel_err(lad.cpu(), g["lad_fp64"]) <= max(3e-5, 3 * rel_err(g["lad"], g["lad_fp64"]))
    before = _native.launch_count()
    xi, li = ar.inverse(x)
    assert _native.launch_count() - before >= 64          # one fused pass per feature
    # the D-step inverse amplifies round-off along the chain: the reference's own fp32 result is ~8e-3 from its fp64 result
    # on these inputs, so the check is the fp64 sandwich
    assert rel_err(xi.cpu(), g["xinv_fp64"]) <= max(1e-4, 3 * rel_err(g["xinv"], g["xinv_fp64"]))
    assert rel_err(li.cpu(), g["ladinv_fp64"]) <= max(1e-3, 3 * rel_err(g["ladinv"], g["ladinv_fp64"]))
    # (no forward->inverse round trip here: with log|det| ~ -30 the inverse expands round-off of y by many orders of
    # magnitude -- the reference's own fp64 round trip is off by O(1) on these weights)
    # FFMA / unfused route gives the same answer
    config.fuse_coupling = False
    try:
        y2, lad2 = ar(x)
    finally:
        config.fuse_coupling = True
    # (two of our own routes: each is held to the fp64 sandwich; against each other only loosely -- sharp bins amplify the
    # last-bit differences of the two dense-layer schedules)
    assert rel_err(y2.cpu(), g["y_fp64"]) <= max(TOL, 3 * rel_err(g["y"], g["y_fp64"])) and rel_err(y2, y) <= 5e-5


@torch.no_grad()
def test_fp16_range_overflow_is_handled_not_silent(cuda_device):
    """Activations beyond the fp16 split range (|a| * 2^config.activation_exp > 65000) trip the flag word; the call is then
    repeated with a smaller activation exponent and meets parity (the reference accepts any finite fp32 input).  With
    auto_activation_exp off the overflow raises instead -- never a silently wrong result."""
    from nflows_b200 import kernels as K
    torch.manual_seed(3)
    lu = T.LULinear(16).eval()
    x = torch.randn(64, 16) * 300.0
    x[5, 3] = 4000.0                                    # 4000 * 2^6 overflows fp16
    want = lu(x)[0]
    lu = lu.to(cuda_device)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y, _ = lu(x.to(cuda_device))
    assert rel_err(y.cpu(), want) <= TOL
    assert config.activation_exp == 6                  # the lowered exponent does not outlive the call
    config.auto_activation_exp = False
    try:
        with pytest.raises(K.Float16RangeError):
            lu(x.to(cuda_device))
    finally:
        config.auto_activation_exp = True
    old = config.activation_exp
    config.activation_exp = 2
    try:
        y, _ = lu(x.to(cuda_device))
    finally:
        config.activation_exp = old
    assert rel_err(y.cpu(), want) <= TOL


@torch.no_grad()
def test_flow_on_inputs_of_large_magnitude_matches_the_oracle(cuda_device):
    """A drop-in has no input-magnitude cliff: the NSF flow on x * 1e4 (far outside the spline tails, activations ~1e4..1e6)
    agrees with the CPU oracle."""
    import warnings
    torch.manual_seed(0)
    flow = recipes.perturb_(recipes.rq_nsf(features=64, hidden_features=64, num_layers=3).eval())
    sd = {k: v.clone() for k, v in flow.state_dict().items()}
    x = torch.randn(700, 64) * 1e4
    want = O.flow_log_prob(sd, O.nsf_spec(3), x)
    flow = flow.to(cuda_device)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with native_launches():
            got = flow.log_prob(x.to(cuda_device))
    assert rel_err(got.cpu(), want) <= TOL


@pytest.mark.gpu
@torch.no_grad()
def test_image_flow_against_reference_golden(cuda_device):
    """SURVEY section 8 row f3 / BASELINE cfg 5 in small (tests/golden/image_rows.pt, reference outputs): Glow-style multiscale
    flow on 3x16x16 images.  Every level runs as a pixel-row chain on our kernels -- layout change, squeeze gather, folded
    ActNorm + 1x1 convolution, ConvResidualNet as dense layers (im2col of the fp16 pair for the 3x3 convolutions), fused final
    layer + spline, per-sample log|det| -- forward, log_prob and inverse."""
    g = load_golden("image_rows")["glow_small"]
    flow = recipes.glow_multiscale(image_shape=(3, 16, 16), levels=3, steps=2, hidden_channels=32).eval()
    flow.load_state_dict(g["sd"], strict=True)
    flow = flow.to(cuda_device)
    x = g["x"].to(cuda_device)
    K.TIMELINE = []
    try:
        with native_launches():
            z, lad = flow._transform(x)
        tags = {t[0] for t in K.TIMELINE}
    finally:
        K.TIMELINE = None
    assert {"nchw_to_rows", "rows_to_nchw", "im2col3x3_32", "rq_coupling_final"} <= tags, tags
    assert rel_err(z.cpu(), g["z_fp64"]) <= max(TOL, 3 * rel_err(g["z"], g["z_fp64"]))
    lp = flow.log_prob(x)
    assert rel_err(lp.cpu(), g["log_prob_fp64"]) <= max(TOL, 3 * rel_err(g["log_prob"], g["log_prob_fp64"]))
    xs, lad_inv = flow._transform.inverse(g["noise"].to(cuda_device))
    assert rel_err(xs.cpu(), g["sample_fp64"]) <= max(1e-4, 3 * rel_err(g["sample"], g["sample_fp64"]))
    assert rel_err(lad_inv.cpu(), g["lad_inv_fp64"]) <= max(1e-4, 3 * rel_err(g["lad_inv"], g["lad_inv_fp64"]))
    # batch split consistency: images are independent
    lp2 = torch.cat([flow.log_prob(x[:2]), flow.log_prob(x[2:])])
    assert rel_err(lp2.cpu(), lp.cpu()) <= 1e-6
    assert flow.sample(3).shape == (3, 3, 16, 16)


@torch.no_grad()
def test_affine_couplings_fused_final_layer_against_reference_golden(cuda_device):
    """Row ns2 (north_star: AffineCouplingTransform gets the same fused treatment): the last conditioner layer and the affine /
    additive coupling run as ONE tcgen05 kernel (nfk_affine_coupling_final_f16x3), the trunk before it as one launch of the
    coupling-step kernel stopped after its last trunk layer; reference outputs in tests/golden/affine_rows.pt."""
    from nflows_b200.distributions.normal import StandardNormal
    from nflows_b200.flows import Flow
    g = load_golden("affine_rows")
    f = lambda i, o: ResidualNet(i, o, hidden_features=64, num_blocks=2)
    alt = torchutils.create_alternating_binary_mask
    cases = [("default48", T.AffineCouplingTransform(alt(48), f)),
             ("general48", T.AffineCouplingTransform(alt(48), f, scale_activation=T.AffineCouplingTransform.GENERAL_SCALE_ACTIVATION)),
             ("default20", T.AffineCouplingTransform(torch.tensor([0] * 8 + [1] * 12), f)),
             ("additive48", T.AdditiveCouplingTransform(alt(48), f))]
    for key, t in cases:
        r = g[key]
        t.load_state_dict(r["sd"], strict=True)
        t = to_dev(t, cuda_device)
        x = r["x"].to(cuda_device)
        K.TIMELINE = []
        try:
            with native_launches():
                y, lad = t(x)
            tags = {e[0] for e in K.TIMELINE}
        finally:
            K.TIMELINE = None
        assert "affine_coupling_final" in tags and "trunk_step" in tags, (key, tags)
        idf = t.identity_features.cpu()
        assert torch.equal(y.cpu()[:, idf], r["x"][:, idf]), key
        if "y_fp64" in r:
            assert rel_err(y.cpu(), r["y_fp64"]) <= max(TOL, 3 * rel_err(r["y"], r["y_fp64"])), key
            assert rel_err(lad.cpu(), r["lad_fp64"]) <= max(TOL, 3 * rel_err(r["lad"], r["lad_fp64"])), key
        else:
            assert rel_err(y.cpu(), r["y"]) <= TOL and torch.equal(lad.cpu(), torch.zeros(x.shape[0])), key
        xi, li = t.inverse(x)
        assert rel_err(xi.cpu(), r["xinv"]) <= 1e-4, key
        if "ladinv" in r:
            assert rel_err(li.cpu(), r["ladinv"]) <= 3e-5, key
    r = g["flow48"]
    steps = []
    for i in range(3):
        steps += [T.ActNorm(48), T.CompositeTransform([T.RandomPermutation(48), T.LULinear(48, identity_init=True)]),
                  T.AffineCouplingTransform(alt(48, even=(i % 2 == 0)), f)]
    flow = Flow(T.CompositeTransform(steps), StandardNormal([48])).eval()
    flow.load_state_dict(r["sd"], strict=True)
    flow = flow.to(cuda_device)
    lp = flow.log_prob(r["x"].to(cuda_device))
    assert rel_err(lp.cpu(), r["log_prob_fp64"]) <= max(TOL, 3 * rel_err(r["log_prob"], r["log_prob_fp64"]))
    assert rel_err(flow.transform_to_noise(r["x"].to(cuda_device)).cpu(), r["z"]) <= 5e-5
