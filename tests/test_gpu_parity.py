"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Everything goes through the C ABI.

Stated tolerance (BASELINE.json north_star): per-sample `log_prob` rtol <= 1e-4 against the reference
(fp64 golden / fp64 oracle), with atol 1e-3 for |log_prob| < 10; scalar forward_kld rel 2e-5;
per-layer z atol 2e-4, per-layer log_det atol 2e-3 (fp32 conditioning of single spline elements, see
tests/test_spline_host.py).  The golden vectors were minted from the real reference
(tests/golden/make_golden.py); the oracle (oracle/nf_oracle.py) is pinned to them on CPU."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden
from helpers import annotate_spec, build_model, rel_err
from oracle import nf_oracle as O

import normflows as nf
from normflows.flows.base import NativeFlow

pytestmark = pytest.mark.gpu

CASES = ["nsf_ar_d64_h256_l2", "nsf_ar_d5_h128_l3", "nsf_ar_d2_h32_l2_k4", "nsf_coupled_d64_h256_l2",
         "nsf_coupled_d5_h128_l3", "nsf_coupled_d2_h32_l2_k4", "realnvp2d", "affine_block2d", "affine_block6d"]
RTOL, ATOL = 1e-4, 1e-3


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


@pytest.fixture(autouse=True)
def _tc_default():
    NativeFlow.use_tensor_cores = True
    yield
    NativeFlow.use_tensor_cores = True


@pytest.mark.parametrize("use_tc", [True, False])
@pytest.mark.parametrize("name", CASES)
def test_log_prob_and_kld_match_reference(name, use_tc):
    NativeFlow.use_tensor_cores = use_tc
    spec, sd, a = load_golden(name)
    model = build_model(annotate_spec(spec, sd), sd).cuda()
    x = cuda(a["x"])
    lp = model.log_prob(x).cpu().numpy()
    np.testing.assert_allclose(lp, a["log_prob_f64"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(lp, a["log_prob_f32"], rtol=RTOL, atol=ATOL)
    kld = float(model.forward_kld(x))
    assert kld == pytest.approx(float(a["kld_f64"]), rel=2e-5)
    if use_tc and "d64" in name:
        assert model._stack().fused_layers() == list(range(len(model.flows))), "flagship shape must run fused"


@pytest.mark.parametrize("use_tc", [True, False])
@pytest.mark.parametrize("name", CASES)
def test_per_layer_inverse_matches_reference(name, use_tc):
    NativeFlow.use_tensor_cores = use_tc
    spec, sd, a = load_golden(name)
    model = build_model(annotate_spec(spec, sd), sd).cuda()
    n = len(model.flows)
    for i in range(n - 1, -1, -1):
        zin = a["x"] if i == n - 1 else a[f"zl_f64__{i + 1}"]
        z, ld = model.flows[i].inverse(cuda(zin))
        assert z.dtype == torch.float32 and ld.shape == (zin.shape[0],)
        np.testing.assert_allclose(z.cpu().numpy(), a[f"zl_f64__{i}"], rtol=1e-4, atol=2e-4, err_msg=f"layer {i}")
        np.testing.assert_allclose(ld.cpu().numpy(), a[f"ld_f64__{i}"], rtol=1e-4, atol=2e-3, err_msg=f"layer {i}")


@pytest.mark.parametrize("name", [c for c in CASES if c != "nsf_ar_d64_h256_l2"])
def test_sampling_direction_matches_reference(name):
    spec, sd, a = load_golden(name)
    model = build_model(annotate_spec(spec, sd), sd).cuda()
    xr, ld = model.forward_and_log_det(cuda(a["z_f64"]))
    # The sampling direction is ill-conditioned for a few rows whose latents sit far in the tails
    # (autoregressive inverse = D chained spline inversions): the reference's OWN fp32 run differs from
    # its fp64 run by up to 7.6e-2 there (tests/golden: fwd_x_f32 vs fwd_x_f64).  Bound the bulk tightly
    # and the tail by the reference's fp32 spread.
    ex = np.abs(xr.cpu().numpy() - a["fwd_x_f64"]).max(axis=1)
    ref_spread = np.abs(a["fwd_x_f32"] - a["fwd_x_f64"]).max()
    assert np.median(ex) < 2e-4 and np.mean(ex < 1e-3) >= 0.8, np.sort(ex)[-5:]
    assert ex.max() <= max(10 * ref_spread, 2e-3), (ex.max(), ref_spread)
    el = np.abs(ld.cpu().numpy() - a["fwd_ld_f64"])
    ref_spread_l = np.abs(a["fwd_ld_f32"] - a["fwd_ld_f64"]).max()
    assert np.median(el) < 2e-3 and np.mean(el < 1e-2) >= 0.8 and el.max() <= max(10 * ref_spread_l, 2e-2), (el.max(), ref_spread_l)


def test_inverse_and_log_det_and_round_trip_ar64():
    spec, sd, a = load_golden("nsf_ar_d64_h256_l2")
    model = build_model(spec, sd).cuda()
    z, ld = model.inverse_and_log_det(cuda(a["x"]))
    # single latent elements that land on a steep spline segment move by a few 1e-4 in fp32 (see
    # tests/test_spline_host.py); bound the bulk tightly and every element loosely
    ez = np.abs(z.cpu().numpy() - a["z_f64"])
    assert np.mean(ez < 2e-4) > 0.995 and ez.max() < 2e-3, ez.max()
    # sampling direction of the autoregressive layer = D sequential MADE passes
    xr, ld2 = model.forward_and_log_det(z)
    # 64 chained spline inversions per layer amplify fp32 round-off on a few elements (same in the reference)
    ex = np.abs(xr.cpu().numpy() - a["x"])
    assert np.mean(ex < 2e-3) > 0.998 and ex.max() < 0.1, ex.max()
    assert np.median(np.abs((ld + ld2).cpu().numpy())) < 2e-2


def _random_model(kind, d=64, layers=4, hidden=256, seed=0, sigma=0.05):
    torch.manual_seed(seed)
    fl = []
    for i in range(layers):
        if kind == "ar":
            fl.append(nf.flows.AutoregressiveRationalQuadraticSpline(d, 2, hidden))
        else:
            fl.append(nf.flows.CoupledRationalQuadraticSpline(d, 2, hidden, reverse_mask=bool(i % 2)))
        fl.append(nf.flows.LULinearPermute(d))
    m = nf.NormalizingFlow(nf.distributions.DiagGaussian(d, trainable=False), fl)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=g))
    return m


def _oracle_of(model, spec_kind, d, layers, hidden):
    sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    flows = []
    for i in range(layers):
        flows.append({"type": "AutoregressiveRationalQuadraticSpline" if spec_kind == "ar"
                      else "CoupledRationalQuadraticSpline", "num_bins": 8, "tail_bound": 3.0})
        flows.append({"type": "LULinearPermute"})
    return {"kind": "NormalizingFlow", "q0": {"shape": [d]}, "flows": flows}, sd


@pytest.mark.parametrize("kind", ["ar", "coupled"])
def test_full_batch_properties(kind):
    """BASELINE batch size (65 536 + a ragged tail): fused kernel vs plain-fp32 kernels on every row,
    a row subset vs the fp64 oracle, run-to-run determinism, and ragged/tiny batches."""
    d, layers, hidden = 64, 4, 256
    model = _random_model(kind, d, layers, hidden).cuda()
    spec, sd = _oracle_of(model, kind, d, layers, hidden)
    B = 65536 + 77
    x = torch.randn(B, d, generator=torch.Generator().manual_seed(1234)) * 1.5
    xc = x.cuda()
    lp = model.log_prob(xc)
    lp2 = model.log_prob(xc)
    assert torch.equal(lp, lp2), "fused path must be deterministic"
    NativeFlow.use_tensor_cores = False
    lp_fp32 = model.log_prob(xc)
    NativeFlow.use_tensor_cores = True
    lpn, lp32n = lp.cpu().numpy().astype(np.float64), lp_fp32.cpu().numpy().astype(np.float64)
    disc = np.abs(lpn - lp32n) / (np.abs(lp32n) + 1e-12)
    assert np.mean(disc < RTOL) > 0.9995 and disc.max() < 5e-4, disc.max()  # two fp32 paths, neither is truth
    idx = np.r_[0:96, 65500:B]
    ref = O.log_prob(spec, sd, x.numpy()[idx].astype(np.float64))
    np.testing.assert_allclose(lpn[idx], ref, rtol=RTOL, atol=ATOL)
    # the tensor core accumulates with truncation; the packer compensates it (nfb_api.cu kAccStepGain).  Pin
    # the residual: uncompensated, the median signed error of this stack is +1.2e-3 (ar) / +0.75e-3 (coupled).
    assert abs(np.median(lpn[idx] - ref)) < 4e-4, np.median(lpn[idx] - ref)
    # the rows where the two GPU paths disagree most: judge each against fp64 truth, relative to what the
    # reference's own fp32 arithmetic (the oracle run in float32) loses on the very same rows
    worst = np.argsort(disc)[-24:]
    truth = O.log_prob(spec, sd, x.numpy()[worst].astype(np.float64))
    ref32 = O.log_prob(spec, sd, x.numpy()[worst].astype(np.float32)).astype(np.float64)
    e_ref32 = np.abs(ref32 - truth) / np.abs(truth)
    e_fused = np.abs(lpn[worst] - truth) / np.abs(truth)
    # Split-bf16 products carry ~2^-17 relative error (vs 2^-24 for fp32 FMAs).  Over 65 613 rows of this
    # deliberately rough model (sigma 0.05, 4 blocks) the WORST rows reach ~1.4e-4; 99.95 % of all rows are
    # inside 1e-4 (asserted above on `disc`), the goldens at ~1e-5.  Bound the tail at 3e-4.
    assert e_fused.max() < 3e-4, (e_fused.max(), e_ref32.max())
    assert np.median(e_fused) < RTOL
    for b in (1, 127, 128, 129, 300):
        np.testing.assert_allclose(model.log_prob(xc[:b]).cpu().numpy(), lp.cpu().numpy()[:b], rtol=1e-6, atol=1e-5)
    assert model.log_prob(xc[:0]).shape == (0,)
    assert float(model.forward_kld(xc)) == pytest.approx(-float(lp.double().mean()), rel=1e-6)


def test_sampling_direction_fused_coupled_stack():
    """Coupling-layer stacks run the sampling direction (core.py:40-55) through the same persistent kernel:
    units of [inverse LU map of the previous layer + block with its splines inverted]."""
    spec, sd, a = load_golden("nsf_coupled_d64_h256_l2")
    model = build_model(annotate_spec(spec, sd), sd).cuda()
    n = len(model.flows)
    # per layer: forward of layer i maps the golden's state i to state i+1 with log-det -ld_i
    for i in range(n):
        zout_ref = a["x"] if i == n - 1 else a[f"zl_f64__{i + 1}"]
        z, ld = model.flows[i].forward(cuda(a[f"zl_f64__{i}"]))
        np.testing.assert_allclose(z.cpu().numpy(), zout_ref, rtol=1e-4, atol=1e-3, err_msg=f"layer {i}")
        np.testing.assert_allclose(ld.cpu().numpy(), -a[f"ld_f64__{i}"], rtol=1e-4, atol=5e-3, err_msg=f"layer {i}")
    xr, ld = model.forward_and_log_det(cuda(a["z_f64"]))
    assert model._stack().launch_count() <= 8, "coupled stack must sample through the whole-stack launch"
    np.testing.assert_allclose(xr.cpu().numpy(), a["fwd_x_f64"], rtol=1e-4, atol=2e-3)
    np.testing.assert_allclose(ld.cpu().numpy(), a["fwd_ld_f64"], rtol=1e-4, atol=2e-2)

    # BASELINE batch size: fused sampling vs the plain-fp32 kernels on every row, vs the fp64 oracle on a
    # subset, and the round trip x -> z -> x through both fused directions
    d, layers, hidden = 64, 4, 256
    model = _random_model("coupled", d, layers, hidden).cuda()
    spec, sd = _oracle_of(model, "coupled", d, layers, hidden)
    B = 65536 + 77
    x = (torch.randn(B, d, generator=torch.Generator().manual_seed(99)) * 1.5).cuda()
    z, ld_inv = model.inverse_and_log_det(x)
    x2, ld_fwd = model.forward_and_log_det(z)
    x2b, _ = model.forward_and_log_det(z)
    assert torch.equal(x2, x2b), "fused sampling path must be deterministic"
    ex = (x2 - x).abs().max(dim=1).values.cpu().numpy()
    assert np.mean(ex < 5e-4) > 0.995 and ex.max() < 5e-2, (np.mean(ex < 5e-4), ex.max())
    assert np.median(np.abs((ld_inv + ld_fwd).cpu().numpy())) < 2e-3
    NativeFlow.use_tensor_cores = False
    x32, ld32 = model.forward_and_log_det(z)
    NativeFlow.use_tensor_cores = True
    dx = (x2 - x32).abs().max(dim=1).values.cpu().numpy()
    assert np.mean(dx < 5e-4) > 0.995 and dx.max() < 5e-2, (np.mean(dx < 5e-4), dx.max())
    idx = np.r_[0:64, B - 40:B]
    zo = z.cpu().numpy()[idx].astype(np.float64)
    xo, ldo = O.forward_and_log_det(spec, sd, zo)
    e = np.abs(x2.cpu().numpy()[idx] - xo).max(axis=1)
    assert np.median(e) < 2e-4 and e.max() < 2e-2, np.sort(e)[-4:]
    el = np.abs(ld_fwd.cpu().numpy()[idx] - ldo)
    assert np.median(el) < 2e-3 and el.max() < 5e-2, np.sort(el)[-4:]


def test_edge_inputs_through_fused_kernel():
    """x exactly at +-B, just outside, far outside and NaN (SURVEY 8c.4) through the fused block."""
    spec, sd, a = load_golden("nsf_ar_d64_h256_l2")
    model = build_model(spec, sd).cuda()
    x = a["x"].copy()
    x[0, :4] = [3.0, -3.0, 3.0000002, -3.0000002]
    x[1, :3] = [100.0, -1e6, 0.0]
    layer = model.flows[2]
    z, ld = layer.inverse(cuda(x))
    zo, ldo = O.ar_rqs(x.astype(np.float64), O._cast(sd, np.float64), "flows.2.", spec["flows"][2], "inverse")
    np.testing.assert_allclose(z.cpu().numpy(), zo, rtol=1e-4, atol=2e-4)
    np.testing.assert_allclose(ld.cpu().numpy(), ldo, rtol=1e-4, atol=2e-3)
    assert z[0, 2].item() == np.float32(3.0000002) and z[1, 0].item() == 100.0 and z[1, 1].item() == -1e6
    xn = cuda(x)
    xn[5, 7] = float("nan")
    zn, ldn = layer.inverse(xn)
    assert torch.isnan(zn[5, 7]) and torch.isfinite(zn[4]).all()


def test_standalone_spline_kernel_edges():
    import ctypes as C
    from normflows import _lib as L
    f = np.load(os.path.join(GOLDEN, "spline_edges.npz"))
    x = cuda(f["x_f32"].reshape(-1, 1))
    params = cuda(np.concatenate([f["uw_f32"], f["uh_f32"], f["ud_f32"]], axis=1))
    for inv in (0, 1):
        y, ld = torch.empty_like(x), torch.empty(x.shape[0], device="cuda")
        L.check(L.lib().nfb_rqs_spline(L.ptr(x), L.ptr(params), L.ptr(y), L.ptr(ld), x.shape[0], 1, 8,
                                       C.c_float(3.0), C.c_float(1.0), inv, 0, None))
        np.testing.assert_allclose(y.cpu().numpy()[:, 0], f[f"y_f64_{inv}"], rtol=1e-5, atol=2e-5, equal_nan=True)
        np.testing.assert_allclose(ld.cpu().numpy(), f[f"lad_f64_{inv}"], rtol=1e-4, atol=5e-4, equal_nan=True)


def test_host_entry_points_and_repack():
    spec, sd, a = load_golden("nsf_coupled_d64_h256_l2")
    model = build_model(spec, sd).cuda()
    xh = torch.from_numpy(a["x"].astype(np.float32)).pin_memory()
    lp_host = model.log_prob_host(xh)
    np.testing.assert_allclose(lp_host.numpy(), a["log_prob_f64"], rtol=RTOL, atol=ATOL)
    assert model.forward_kld_host(xh) == pytest.approx(float(a["kld_f64"]), rel=2e-5)
    # parameter update -> packed weights must follow (cache invalidation by tensor version)
    with torch.no_grad():
        model.flows[0].prqct.transform_net.final_layer.bias.add_(0.1)
    sd2 = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    ref = O.log_prob(spec, sd2, a["x"].astype(np.float64))
    np.testing.assert_allclose(model.log_prob(cuda(a["x"])).cpu().numpy(), ref, rtol=RTOL, atol=ATOL)


def test_actnorm_data_dependent_init():
    f = np.load(os.path.join(GOLDEN, "actnorm_init.npz"))
    an = nf.flows.ActNorm(6).cuda()
    x = f["x"][:, :, 0, 0]  # [8, 6] slice as a 2-D batch
    z, ld = an.inverse(cuda(x))
    s, t = O.actnorm_init(x.astype(np.float64), (1, 6), "inverse")
    np.testing.assert_allclose(an.s.detach().cpu().numpy(), s, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(an.t.detach().cpu().numpy(), t, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(z.cpu().numpy(), (x - t) * np.exp(-s), rtol=1e-4, atol=1e-5)
    assert float(an.data_dep_init_done) == 1.0


def test_glow_multiscale_log_prob_matches_reference():
    """SURVEY 8a rows a2/a13-a17 on images: GlowBlock (ConvNet2d coupling + Invertible1x1Conv + ActNorm),
    Squeeze, channel split, ClassCondDiagGaussian, MultiscaleFlow.log_prob / forward_kld."""
    from helpers_glow import build_glow_small
    spec, sd, a = load_golden("glow_small")
    model = build_glow_small(sd).cuda()
    x = cuda(a["x"])
    y = torch.from_numpy(a["y"]).cuda()
    lp = model.log_prob(x, y).cpu().numpy()
    np.testing.assert_allclose(lp, a["log_prob_f64"], rtol=RTOL, atol=ATOL)
    assert float(model.forward_kld(x, y)) == pytest.approx(float(a["kld_f64"]), rel=2e-5)
    # one block against the oracle, with its log-det
    z0 = np.random.default_rng(3).normal(size=(5, 24, 2, 2))
    blk = model.flows[0][0]
    z, ld = blk.inverse(cuda(z0))
    zo, ldo = O.glow_block(z0, O._cast(sd, np.float64), "flows.0.0.", {}, "inverse")
    np.testing.assert_allclose(z.cpu().numpy(), zo, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(ld.cpu().numpy(), ldo, rtol=1e-4, atol=1e-3)
    # squeeze round trip + oracle
    s = nf.flows.Squeeze()
    zs, _ = s.inverse(cuda(a["x"]))
    np.testing.assert_array_equal(zs.cpu().numpy(), O.squeeze(a["x"].astype(np.float32), None, "", {}, "inverse")[0])
    zr, _ = s.forward(zs)
    np.testing.assert_array_equal(zr.cpu().numpy(), a["x"].astype(np.float32))


def test_glow_sampling_direction_matches_reference():
    """Rows a2/a13/a14 in the sampling direction (core.py:504-525, glow.py:72-77, mixing.py:106-121 with the
    double-precision inverse of :94-101): per-level latents from the reference -> x, one block, round trip."""
    from helpers_glow import build_glow_small
    spec, sd, a = load_golden("glow_small")
    model = build_glow_small(sd).cuda()
    n = len(spec["levels"])
    zs = [cuda(a[f"ms_z{j}_f64"]) for j in range(n)]
    x, ld = model.forward_and_log_det(zs)
    np.testing.assert_allclose(x.cpu().numpy(), a["ms_fwd_x_f64"], rtol=1e-4, atol=2e-4)
    np.testing.assert_allclose(ld.cpu().numpy(), a["ms_fwd_ld_f64"], rtol=1e-4, atol=2e-2)
    # our own inverse -> forward round trip on the golden images
    zl, ld_inv = model.inverse_and_log_det(cuda(a["x"]))
    for j in range(n):
        np.testing.assert_allclose(zl[j].cpu().numpy(), a[f"ms_z{j}_f64"], rtol=1e-4, atol=5e-4)
    np.testing.assert_allclose(ld_inv.cpu().numpy(), a["ms_inv_ld_f64"], rtol=1e-4, atol=2e-2)
    xr, ld_fwd = model.forward_and_log_det(zl)
    np.testing.assert_allclose(xr.cpu().numpy(), a["x"], rtol=1e-4, atol=5e-4)
    assert np.abs((ld_inv + ld_fwd).cpu().numpy()).max() < 2e-2
    # one block against the oracle, with its log-det
    z0 = np.random.default_rng(4).normal(size=(5, 24, 2, 2))
    blk = model.flows[0][0]
    z, ldb = blk.forward(cuda(z0))
    zo, ldo = O.glow_block(z0, O._cast(sd, np.float64), "flows.0.0.", {}, "forward")
    np.testing.assert_allclose(z.cpu().numpy(), zo, rtol=1e-4, atol=2e-4)
    np.testing.assert_allclose(ldb.cpu().numpy(), ldo, rtol=1e-4, atol=1e-3)
    # sampling: shapes, finiteness, and log_q consistent with the density of what was drawn
    y = torch.from_numpy(a["y"]).cuda()
    torch.manual_seed(7)
    xs, lq = model.sample(len(y), y)
    assert xs.shape == (len(y), 3, 8, 8) and torch.isfinite(xs).all() and torch.isfinite(lq).all()
    np.testing.assert_allclose(lq.cpu().numpy(), model.log_prob(xs, y).cpu().numpy(), rtol=1e-4, atol=2e-2)


@pytest.mark.parametrize("shape", [
    # (B, ctot, c0, cin, H, W, cout, ks, leaky)   Glow conditioner shapes (nets/cnn.py:33-61) + awkward ones
    (5, 12, 0, 6, 16, 16, 256, 3, 0.0),      # first conv, level 1: K = 54 (one padded chunk), N = 256
    (3, 256, 0, 256, 8, 8, 256, 1, 0.0),     # middle 1x1 conv: K = 256 (4 chunks)
    (3, 256, 0, 256, 8, 8, 24, 3, -1.0),     # last conv: K = 2304 (36 chunks), N = 24 -> 32, no activation
    (37, 48, 24, 24, 4, 4, 256, 3, 0.1),     # 4x4 images: a 128-pixel tile spans 8 images; channel slice; ragged M
    (2, 7, 1, 5, 5, 7, 200, 5, 0.0),         # odd everything, 5x5 kernel, N = 200 -> 208
    (9, 12, 0, 12, 16, 16, 12, 1, -1.0),     # folded ActNorm + 1x1 conv: small-channel fp32 kernel
    (4, 50, 1, 48, 4, 4, 48, 1, -1.0),
])
def test_conv2d_tensor_core_matches_oracle(shape):
    """nfb_conv2d routes conditioner-sized convolutions to the tcgen05 implicit-GEMM kernel (csrc/nfb_conv_tc.cu)."""
    from normflows import _lib as L
    B, ctot, c0, cin, H, W, cout, ks, leaky = shape
    rng = np.random.default_rng(sum(shape[:8]))
    x = rng.normal(size=(B, ctot, H, W)).astype(np.float32)
    w = (rng.normal(size=(cout, cin, ks, ks)) / np.sqrt(cin * ks * ks)).astype(np.float32)
    b = rng.normal(size=cout).astype(np.float32)
    ref = O.conv2d(x[:, c0:c0 + cin].astype(np.float64), w.astype(np.float64), b.astype(np.float64))
    if leaky >= 0:
        ref = np.where(ref >= 0, ref, ref * leaky)
    xd, wd, bd = cuda(x), cuda(w), cuda(b)
    y = torch.full((B, cout, H, W), float("nan"), device="cuda")
    L.check(L.lib().nfb_conv2d(L.ptr(xd), ctot, c0, L.ptr(wd), L.ptr(bd), L.ptr(y), B, cin, H, W, cout, ks,
                               float(leaky), L.stream_ptr()))
    got = y.cpu().numpy()
    assert np.isfinite(got).all()
    # split-bf16 products: ~2^-17 relative per term, K terms of unit scale
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=2e-5 * np.sqrt(cin * ks * ks))
    assert np.abs(np.mean(got - ref)) < 3e-6  # no one-sided accumulate bias left


def test_glow_actnorm_data_dependent_init_on_images():
    f = np.load(os.path.join(GOLDEN, "actnorm_init.npz"))
    blk = nf.flows.GlowBlock(6, 8).cuda()
    z, ld = blk.inverse(cuda(f["x"]))  # first call initialises ActNorm from the batch (normalization.py:33-38)
    an = blk.flows[2]
    np.testing.assert_allclose(an.s.detach().cpu().numpy(), f["s"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(an.t.detach().cpu().numpy(), f["t"], rtol=1e-5, atol=1e-6)
    assert float(an.data_dep_init_done) == 1.0 and torch.isfinite(z).all() and torch.isfinite(ld).all()


@pytest.mark.parametrize("kind", ["ar", "coupled"])
def test_backward_matches_reference_gradients(kind):
    """loss.backward() (examples/neural_spline_flow.ipynb cell 4): forward value from the CUDA kernels,
    gradients from the interim autograd hook (normflows/_autograd.py) vs gradients minted from the reference."""
    spec, sd, _ = load_golden(f"nsf_{kind}_d5_h128_l3")
    g = np.load(os.path.join(GOLDEN, f"grads_nsf_{kind}_d5_h128_l3.npz"))
    model = build_model(spec, sd).cuda()
    torch.set_grad_enabled(True)  # (the autouse fixture restores the previous mode)
    for p in model.parameters():
        p.requires_grad_(True)
    x = cuda(g["x"]).requires_grad_(True)
    loss = model.forward_kld(x)
    assert float(loss.detach()) == pytest.approx(float(g["kld"]), rel=2e-5)
    loss.backward()
    np.testing.assert_allclose(x.grad.cpu().numpy(), g["grad__x"], rtol=2e-3, atol=2e-5)
    checked = 0
    for k, p in model.named_parameters():
        if "grad__" + k in g.files:
            ref = g["grad__" + k]
            assert p.grad is not None, k
            scale = np.abs(ref).max() + 1e-8
            assert np.abs(p.grad.cpu().numpy() - ref).max() <= 2e-3 * scale + 1e-6, k
            checked += 1
    assert checked > 20
    # the usual training step works end to end
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    opt.step()
    assert torch.isfinite(model.forward_kld(x.detach()).detach()).item()  # packed weights follow the update


# ---------------------------------------------------------------------------------------------------------
# Parity ON THE BENCHMARKED CONFIGURATION (BASELINE.json configs[1]; bench.build_model): 32 layers, d=64,
# hidden 256, B = 65 536 + a ragged tail.  Stated tolerance, no crutches: per-sample log_prob rtol 1e-4 against
# the fp64 oracle on EVERY checked row (first tiles, last/ragged tiles, random rows, and the rows where the
# fused path differs most from the plain-fp32 kernels over the whole batch); forward_kld rel 2e-5.
# ---------------------------------------------------------------------------------------------------------
def _bench_module():
    import importlib
    import sys
    from conftest import ROOT
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    return importlib.import_module("bench")


@pytest.mark.parametrize("kind", ["ar", "coupled"])
def test_bench_config_32_layers_parity(kind):
    bench = _bench_module()
    model = bench.build_model(kind).cuda()
    spec = bench.oracle_spec(kind)
    sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    B = 65536 + 77
    x = torch.randn(B, 64, generator=torch.Generator().manual_seed(1234)) * 1.5
    xc = x.cuda()
    lp = model.log_prob(xc)
    assert model._stack().fused_layers() == list(range(64)), "bench stack must run on the fused tcgen05 kernel"
    assert model._stack().launch_count() <= 8
    NativeFlow.use_tensor_cores = False
    lp32 = model.log_prob(xc)
    NativeFlow.use_tensor_cores = True
    lpn, lp32n = lp.cpu().numpy().astype(np.float64), lp32.cpu().numpy().astype(np.float64)
    assert np.isfinite(lpn).all()
    disc = np.abs(lpn - lp32n) / np.abs(lp32n)
    rng = np.random.default_rng(5)
    idx = np.unique(np.r_[0:256, B - 333:B, rng.integers(0, B, 1200), np.argsort(disc)[-256:]])
    truth = O.log_prob(spec, sd, x.numpy()[idx].astype(np.float64))
    rel = np.abs(lpn[idx] - truth) / np.abs(truth)
    rel32 = np.abs(lp32n[idx] - truth) / np.abs(truth)
    print(f"\n[{kind}] 32 layers, {len(idx)} rows vs fp64: fused rel max {rel.max():.2e} p99 {np.quantile(rel, .99):.2e} "
          f"median {np.median(rel):.2e} | signed mean {np.mean(lpn[idx] - truth):+.2e} | plain-fp32 kernels rel max "
          f"{rel32.max():.2e} | fused-vs-fp32 over all {B} rows: max {disc.max():.2e}, >1e-4: {int((disc > 1e-4).sum())}")
    assert rel.max() < RTOL, (rel.max(), idx[np.argmax(rel)])          # every checked row, no atol
    assert rel32.max() < RTOL
    assert disc.max() < 2 * RTOL                                        # all 65 613 rows: the two GPU paths agree
    kld = float(model.forward_kld(xc))
    assert kld == pytest.approx(-float(lpn.mean()), rel=1e-6)
    # scalar loss against fp64 on the checked rows (same rows on both sides)
    assert -lpn[idx].mean() == pytest.approx(-truth.mean(), rel=2e-5)


@pytest.mark.parametrize("kind", ["ar", "coupled"])
def test_trained_weights_parity(kind):
    """Weights TRAINED with the reference (tests/golden/make_trained.py: 400 Adam steps of forward_kld on a
    structured 64-d target) -- off the calibration set of the accumulate-truncation compensation (kAccStepGain):
    post-ReLU activations against correlated weights.  log_prob rtol 1e-4 on every row vs the reference's fp64."""
    import json
    f = np.load(os.path.join(GOLDEN, f"trained_{kind}_d64_h256_l4.npz"))
    meta = json.loads(str(f["meta"]))
    torch.manual_seed(meta["seed"])  # masks / permutations are functions of the constructor seed
    fl = []
    for i in range(meta["layers"]):
        if kind == "ar":
            fl.append(nf.flows.AutoregressiveRationalQuadraticSpline(64, 2, meta["hidden"]))
        else:
            fl.append(nf.flows.CoupledRationalQuadraticSpline(64, 2, meta["hidden"], reverse_mask=bool(i % 2)))
        fl.append(nf.flows.LULinearPermute(64))
    model = nf.NormalizingFlow(nf.distributions.DiagGaussian(64, trainable=False), fl)
    params = dict(model.named_parameters())
    with torch.no_grad():
        for k in f.files:
            if k.startswith("sd__"):
                params[k[4:]].copy_(torch.from_numpy(f[k]))
    assert sum(1 for k in f.files if k.startswith("sd__")) == len(params)
    model = model.cuda()
    lp = model.log_prob(cuda(f["x"])).cpu().numpy().astype(np.float64)
    assert model._stack().fused_layers() == list(range(2 * meta["layers"]))
    rel = np.abs(lp - f["log_prob_f64"]) / np.abs(f["log_prob_f64"])
    rel_ref32 = np.abs(f["log_prob_f32"] - f["log_prob_f64"]) / np.abs(f["log_prob_f64"])
    print(f"\n[trained {kind}] rel max {rel.max():.2e} median {np.median(rel):.2e} signed mean "
          f"{np.mean(lp - f['log_prob_f64']):+.2e}; the reference's own fp32 run: rel max {rel_ref32.max():.2e}")
    assert rel.max() < RTOL
    assert abs(np.mean(lp - f["log_prob_f64"])) < 2e-4 * np.mean(np.abs(f["log_prob_f64"])) / 10  # no one-sided bias
    assert float(model.forward_kld(cuda(f["x"]))) == pytest.approx(float(f["kld_f64"]), rel=2e-5)


def test_autoregressive_sampling_fused_d64():
    """Sampling direction of the autoregressive block at the flagship shape (flows/affine/autoregressive.py:29-38:
    D = 64 sequential conditioner passes) runs INSIDE the fused tcgen05 unit (one launch for the stack), pinned to
    reference vectors minted by tests/golden/make_golden.py ar64fwd.  The reference's own fp32 run differs from its
    fp64 run by 2.8e-4 on these latents (64 chained spline inversions per layer); bound ours by the same spread."""
    spec, sd, _ = load_golden("nsf_ar_d64_h256_l2")
    f = np.load(os.path.join(GOLDEN, "nsf_ar_d64_h256_l2_fwd.npz"))
    model = build_model(spec, sd).cuda()
    z = cuda(f["z_f64"])
    y0, ld0 = model.flows[0].forward(z)   # one autoregressive layer alone
    spread0 = max(np.abs(f["l0_fwd_x_f32"] - f["l0_fwd_x_f64"]).max(), 1e-5)
    e0 = np.abs(y0.cpu().numpy() - f["l0_fwd_x_f64"])
    # 64 chained spline inversions amplify fp32 round-off on a few elements (the reference's own fp32 run: spread0)
    assert np.median(e0) < 1e-5 and e0.max() < max(8 * spread0, 2e-4), (np.median(e0), e0.max(), spread0)
    np.testing.assert_allclose(ld0.cpu().numpy(), f["l0_fwd_ld_f64"], rtol=1e-4, atol=20 * spread0)
    x, ld = model.forward_and_log_det(z)
    assert model._stack().launch_count() <= 8, "autoregressive stack must sample through the whole-stack launch"
    spread = np.abs(f["fwd_x_f32"] - f["fwd_x_f64"]).max()
    ex = np.abs(x.cpu().numpy() - f["fwd_x_f64"])
    print(f"\\n[ar sampling d64] |x - ref64| median {np.median(ex):.2e} max {ex.max():.2e}; reference fp32 spread {spread:.2e}")
    assert np.median(ex) < 2e-5 and ex.max() < max(8 * spread, 1e-3), (np.median(ex), ex.max(), spread)
    spread_l = np.abs(f["fwd_ld_f32"] - f["fwd_ld_f64"]).max()
    el = np.abs(ld.cpu().numpy() - f["fwd_ld_f64"])
    assert np.median(el) < 2e-3 and el.max() < max(8 * spread_l, 2e-2), (np.median(el), el.max(), spread_l)
    # deterministic, and consistent with the density pass of what was produced
    x2, _ = model.forward_and_log_det(z)
    assert torch.equal(x, x2)
    zr, ldr = model.inverse_and_log_det(x)
    assert np.median(np.abs((ld + ldr).cpu().numpy())) < 5e-3


def test_reverse_kld_value():
    """core.py:104-131 on the CUDA path: value against the oracle evaluated on the very samples that were drawn."""
    spec, sd, _ = load_golden("nsf_coupled_d5_h128_l3")
    model = build_model(annotate_spec(spec, sd), sd).cuda()

    class Target(torch.nn.Module):
        def log_prob(self, z):
            return -0.5 * (z ** 2).sum(1) - 0.5 * z.shape[1] * np.log(2 * np.pi)
    model.p = Target()
    torch.manual_seed(11)
    z0, _ = model.q0(512)
    torch.manual_seed(11)
    rk = float(model.reverse_kld(512))
    x, ldo = O.forward_and_log_det(spec, sd, z0.cpu().numpy().astype(np.float64))
    lq0 = O.diag_gaussian_log_prob(z0.cpu().numpy().astype(np.float64), O._cast(sd, np.float64), "q0.")
    ref = np.mean(lq0 - ldo) - np.mean(-0.5 * (x ** 2).sum(1) - 0.5 * x.shape[1] * np.log(2 * np.pi))
    assert rk == pytest.approx(ref, rel=2e-4, abs=2e-3)
    torch.manual_seed(11)
    rk2 = float(model.reverse_kld(512, score_fn=False))
    assert rk2 == pytest.approx(ref, rel=2e-4, abs=5e-3)


def _gemm(A, B, M, N, K, a_mn=0, b_mn=0, **kw):
    import ctypes as C
    from normflows import _lib as L
    d = L.GemmDesc()
    out = kw.pop("out", None)
    Cm = out if out is not None else torch.full((M, N), float("nan"), device="cuda")
    d.A, d.B, d.C = A.data_ptr(), B.data_ptr(), Cm.data_ptr()
    d.lda, d.ldb, d.ldc = A.stride(0), B.stride(0), Cm.stride(0)
    d.M, d.N, d.K, d.a_mn, d.b_mn = M, N, K, a_mn, b_mn
    keep = []
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            keep.append(v)
            setattr(d, k, v.data_ptr())
            if k in ("mask", "mulm"):
                d.ldmask = v.stride(0)
            if k == "resid":
                d.ldres = v.stride(0)
        else:
            setattr(d, k, int(v))
    L.check(L.lib().nfb_gemm_f32(C.byref(d), L.stream_ptr()))
    return Cm


@pytest.mark.parametrize("shape", [
    # (M, N, K): forward X W^T -- both operands K-major
    (300, 256, 256), (1000, 1472, 256), (129, 23, 5), (64, 115, 128), (4096, 64, 64),
    (40000, 512, 192),   # 313 x 2 output tiles on 148 CTAs: several units per CTA (accumulator double-buffering)
])
def test_gemm_tc_forward_layout(shape):
    """csrc/nfb_gemm_tc.cu, K-major x K-major (Y = X W^T + b with the fused epilogues of the training pass)."""
    M, N, K = shape
    g = torch.Generator().manual_seed(M + N + K)
    X = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(N, K, generator=g) / np.sqrt(K)).cuda()
    b = torch.randn(N, generator=g).cuda()
    ref = (X.double() @ W.double().T)
    got = _gemm(X, W, M, N, K)
    np.testing.assert_allclose(got.cpu().numpy(), ref.cpu().numpy(), rtol=1e-4, atol=3e-5)
    # ReLU on load + bias + ReLU-mask + residual + ReLU out
    H = torch.randn(M, N, generator=g).cuda()
    R = torch.randn(M, N, generator=g).cuda()
    got = _gemm(X, W, M, N, K, a_relu=1, bias=b, mask=H, resid=R, relu_out=1)
    ref2 = torch.relu((torch.relu(X).double() @ W.double().T + b.double()) * (H > 0) + R.double())
    np.testing.assert_allclose(got.cpu().numpy(), ref2.cpu().numpy(), rtol=1e-4, atol=3e-5)


@pytest.mark.parametrize("shape", [(300, 64, 1472), (1000, 256, 256), (130, 5, 128), (257, 256, 736)])
def test_gemm_tc_dgrad_layout(shape):
    """gX = gY W: A = gY K-major, B = W [K x N] row-major = MN-major operand (no transpose in memory)."""
    M, N, K = shape
    g = torch.Generator().manual_seed(M * 3 + N + K)
    gY = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(K, N, generator=g) / np.sqrt(K)).cuda()
    got = _gemm(gY, W, M, N, K, b_mn=1)
    ref = gY.double() @ W.double()
    np.testing.assert_allclose(got.cpu().numpy(), ref.cpu().numpy(), rtol=1e-4, atol=3e-5)


@pytest.mark.parametrize("shape", [(200, 70, 5000), (1472, 256, 9000), (256, 64, 70000), (23, 5, 300)])
def test_gemm_tc_wgrad_layout(shape):
    """dW = gY^T X: both operands MN-major (reduction over the batch), split along K with red.global.add."""
    M, N, K = shape
    g = torch.Generator().manual_seed(M + N * 5 + K)
    gY = torch.randn(K, M, generator=g).cuda()
    X = torch.randn(K, N, generator=g).cuda()
    mm = (torch.rand(M, N, generator=g) > 0.5).float().cuda()
    got = _gemm(gY, X, M, N, K, a_mn=1, b_mn=1, b_relu=1, mulm=mm)
    ref = (gY.double().T @ torch.relu(X).double()) * mm.double()
    scale = float(ref.abs().max())
    assert float((got.double() - ref).abs().max()) < 2e-5 * scale + 1e-5
    # accumulate onto an existing gradient
    base = torch.randn(M, N, generator=g).cuda()
    got2 = _gemm(gY, X, M, N, K, a_mn=1, b_mn=1, out=base.clone(), accumulate=1)
    ref2 = base.double() + gY.double().T @ X.double()
    assert float((got2.double() - ref2).abs().max()) < 2e-5 * float(ref2.abs().max()) + 1e-5


def _check_grads(model, g, rtol_scale=2e-3):
    """Compare .grad of every parameter with a golden: whole tensors (`grad__`) or two random projections of a weight
    matrix (`gradv__` = G v, `gradu__` = u G)."""
    checked = 0
    for k, p in model.named_parameters():
        if "grad__" + k in g.files:
            ref = g["grad__" + k]
            assert p.grad is not None, k
            scale = np.abs(ref).max() + 1e-8
            err = np.abs(p.grad.cpu().numpy() - ref).max()
            assert err <= rtol_scale * scale + 1e-6, (k, err, scale)
            checked += 1
        elif "gradv__" + k in g.files:
            assert p.grad is not None, k
            G = p.grad.double().cpu().numpy()
            for got, ref in ((G @ g["projv__" + k], g["gradv__" + k]), (g["proju__" + k] @ G, g["gradu__" + k])):
                scale = np.abs(ref).max() + 1e-8
                assert np.abs(got - ref).max() <= rtol_scale * scale + 1e-6, (k, np.abs(got - ref).max(), scale)
            assert np.linalg.norm(G) == pytest.approx(float(g["gnorm__" + k]), rel=2e-3)
            checked += 1
    return checked


@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("kind", ["ar", "coupled"])
def test_backward_flagship_shape_matches_reference(kind, native):
    """loss.backward() at d=64 / hidden 256 (the fused shape).  native=True: libnfb200's training pass (recompute,
    analytic spline adjoint, dgrad / wgrad on the tensor core -- csrc/nfb_gemm_tc.cu, nfb_backward.cu); native=False:
    the interim torch re-materialisation (kept as the A/B reference).  Both against fp64 autograd of the reference."""
    from normflows._autograd import DensityFn
    spec, sd, _ = load_golden(f"nsf_{kind}_d64_h256_l2")
    g = np.load(os.path.join(GOLDEN, f"grads_nsf_{kind}_d64_h256_l2.npz"))
    model = build_model(spec, sd).cuda()
    torch.set_grad_enabled(True)
    DensityFn.use_native_backward = native
    try:
        for p in model.parameters():
            p.requires_grad_(True)
        x = cuda(g["x"]).requires_grad_(True)
        loss = model.forward_kld(x)
        assert float(loss.detach()) == pytest.approx(float(g["kld"]), rel=2e-5)
        loss.backward()
        gx_ref = g["grad__x"]  # (a handful of elements sit on steep spline segments: bound by the tensor's scale)
        assert np.abs(x.grad.cpu().numpy() - gx_ref).max() <= 2e-3 * np.abs(gx_ref).max() + 1e-6
        assert np.median(np.abs(x.grad.cpu().numpy() - gx_ref)) < 1e-6 + 1e-4 * np.median(np.abs(gx_ref))
        assert _check_grads(model, g) > 20
    finally:
        DensityFn.use_native_backward = True


def test_native_backward_full_batch_and_training_step():
    """1024 + 37 rows (ragged tile) on a 4-layer stack: native gradients against the fp64 gradient oracle
    (oracle/nf_oracle_grad.py, pinned to the reference's autograd) and against the interim autograd; then a few Adam
    steps: the loss goes down and the packed weights follow the update."""
    from normflows._autograd import DensityFn
    from oracle import nf_oracle_grad as G
    torch.set_grad_enabled(True)
    model = _random_model("ar", 64, 4, 256, seed=3, sigma=0.03).cuda()
    spec, sd = _oracle_of(model, "ar", 64, 4, 256)
    xh = torch.randn(1024 + 37, 64, generator=torch.Generator().manual_seed(5)) * 1.2
    x = xh.cuda()
    loss_ref, gref, _ = G.forward_kld_grads(spec, {k: v.astype(np.float64) if v.dtype.kind == "f" else v for k, v in sd.items()},
                                            xh.numpy().astype(np.float64))
    grads = {}
    for native in (True, False):
        DensityFn.use_native_backward = native
        model.zero_grad(set_to_none=True)
        loss = model.forward_kld(x)
        loss.backward()
        grads[native] = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    DensityFn.use_native_backward = True
    assert float(loss.detach()) == pytest.approx(float(loss_ref), rel=2e-5)
    assert len(grads[True]) == len(grads[False]) > 40
    # ReLU kinks: a pre-activation within round-off of zero switches a whole row's contribution on or off, so single
    # entries of a weight gradient can differ by ~1/sqrt(rows) from the fp64 value in ANY fp32-class implementation.
    # (The recompute GEMMs carry ~1e-5 relative error, so a 1061 x 256 activation matrix has a few such flips per layer.)
    # Judge each tensor by the bulk of its entries (>= 97 % within 2e-3 of the scale) and its relative Frobenius error,
    # and bound single entries loosely.
    worst = {True: [0.0, 0.0], False: [0.0, 0.0]}
    for k in grads[True]:
        ref = gref[k]
        scale = float(np.abs(ref).max()) + 1e-8
        for native in (True, False):
            d = grads[native][k].double().cpu().numpy() - ref
            fro = float(np.linalg.norm(d) / (np.linalg.norm(ref) + 1e-12))
            e = float(np.abs(d).max()) / scale
            worst[native] = [max(worst[native][0], fro), max(worst[native][1], e)]
            frac_ok = float(np.mean(np.abs(d) <= 2e-3 * scale))
            assert frac_ok >= 0.97 and fro <= 1e-2 and e <= 5e-2, (k, native, frac_ok, fro, e, scale)
    print(f"\n[grad vs fp64 oracle, 1061 rows] worst (rel. Frobenius, max entry / scale): native {worst[True][0]:.2e}, "
          f"{worst[True][1]:.2e}; interim torch {worst[False][0]:.2e}, {worst[False][1]:.2e}")
    opt = torch.optim.Adam(model.parameters(), lr=2e-4)
    l0 = float(model.forward_kld(x).detach())
    for _ in range(5):
        opt.zero_grad()
        loss = model.forward_kld(x)
        loss.backward()
        opt.step()
    l1 = float(model.forward_kld(x).detach())
    assert np.isfinite(l1) and l1 < l0, (l0, l1)


def _build_glow_options(f):
    L_, K, hidden, shape, ncls = 2, 2, 16, (3, 8, 8), 10
    q0, merges, flows = [], [], []
    for i in range(L_):
        fl = [nf.flows.GlowBlock(shape[0] * 2 ** (L_ + 1 - i), hidden, split_mode="channel", scale=True, use_lu=False,
                                 net_actnorm=True) for _ in range(K)] + [nf.flows.Squeeze()]
        flows += [fl]
        if i > 0:
            merges += [nf.flows.ImageMerge()]
            ls = (shape[0] * 2 ** (L_ - i), shape[1] // 2 ** (L_ - i), shape[2] // 2 ** (L_ - i))
        else:
            ls = (shape[0] * 2 ** (L_ + 1), shape[1] // 2 ** L_, shape[2] // 2 ** L_)
        q0 += [nf.distributions.ClassCondDiagGaussian(ls, ncls)]
    m = nf.MultiscaleFlow(q0, flows, merges, transform=nf.transforms.Logit(0.05))
    sd = {k[4:]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith("sd__")}
    m.load_state_dict(sd, strict=True)
    return m


def test_reference_options_glow_logit_temperature_and_callable_nets():
    """Options of in-scope classes that used to raise (VERDICT r1 missing #7), against vectors minted from the reference
    (tests/golden/make_golden.py options): Invertible1x1Conv(use_lu=False), ConvNet2d(actnorm=True),
    MultiscaleFlow(transform=Logit), temperature-annealed base distributions, nets.* called as modules."""
    f = np.load(os.path.join(GOLDEN, "options.npz"))
    model = _build_glow_options(f).cuda()
    x, y = cuda(f["x"]), torch.from_numpy(f["y"]).cuda()
    lp = model.log_prob(x, y).cpu().numpy()
    np.testing.assert_allclose(lp, f["log_prob_f64"], rtol=RTOL, atol=ATOL)
    for q in model.q0:
        q.temperature = 0.7
    np.testing.assert_allclose(model.log_prob(x, y).cpu().numpy(), f["log_prob_T07_f64"], rtol=RTOL, atol=ATOL)
    model.reset_temperature()
    zl, ld = model.inverse_and_log_det(x)
    np.testing.assert_allclose(ld.cpu().numpy(), f["inv_ld_f64"], rtol=1e-4, atol=2e-2)
    for j in range(2):
        np.testing.assert_allclose(zl[j].cpu().numpy(), f[f"z{j}_f64"], rtol=1e-4, atol=5e-4)
    xr, ldf = model.forward_and_log_det([cuda(f["z0_f64"]), cuda(f["z1_f64"])])
    np.testing.assert_allclose(xr.cpu().numpy(), f["fwd_x_f64"], rtol=1e-4, atol=5e-4)
    np.testing.assert_allclose(ldf.cpu().numpy(), f["fwd_ld_f64"], rtol=1e-4, atol=2e-2)
    torch.manual_seed(3)
    xs, lq = model.sample(8, y[:8], temperature=0.8)   # temperature-annealed sampling runs and is finite
    assert xs.shape == (8, 3, 8, 8) and torch.isfinite(xs).all() and torch.isfinite(lq).all()
    assert all(q.temperature is None for q in model.q0)
    # a stand-alone 1x1 convolution, both parameterisations, round trip
    for use_lu in (False, True):
        conv = nf.flows.Invertible1x1Conv(6, use_lu=use_lu).cuda()
        z0 = torch.randn(4, 6, 5, 5, device="cuda")
        z1, l1 = conv.inverse(z0)
        z2, l2 = conv.forward(z1)
        assert float((z2 - z0).abs().max()) < 1e-4 and abs(float(l1 + l2)) < 1e-3
    # nets called as plain modules
    xin = cuda(f["net_x"])
    nets = {"mlp": nf.nets.MLP([5, 16, 16, 3], leaky=0.1), "mlp_relu": nf.nets.MLP([5, 16, 3]),
            "resnet": nf.nets.ResidualNet(5, 7, 32, num_blocks=2), "made": nf.nets.MADE(5, 32, output_multiplier=3)}
    for name, net in nets.items():
        sd = {k[len(f"net__{name}__"):]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith(f"net__{name}__")}
        net.load_state_dict(sd, strict=True)
        out = net.cuda()(xin).cpu().numpy()
        np.testing.assert_allclose(out, f[f"net_y__{name}"], rtol=1e-4, atol=2e-5, err_msg=name)


def test_neighbour_layers_maf_and_invertible_affine():
    """SURVEY 8f-4: MaskedAffineAutoregressive (one MADE pass forward, D passes inverse) and InvertibleAffine (both
    parameterisations), against vectors minted from the reference (tests/golden/make_golden.py neighbours)."""
    f = np.load(os.path.join(GOLDEN, "neighbours.npz"))
    maf = nf.flows.MaskedAffineAutoregressive(6, 32, num_blocks=2)
    maf.load_state_dict({k[5:]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith("maf__")}, strict=True)
    maf = maf.cuda()
    x = cuda(f["maf_x"])
    y, ld = maf.forward(x)
    np.testing.assert_allclose(y.cpu().numpy(), f["maf_fwd_y"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(ld.cpu().numpy(), f["maf_fwd_ld"], rtol=1e-4, atol=2e-5)
    xi, ldi = maf.inverse(x)
    np.testing.assert_allclose(xi.cpu().numpy(), f["maf_inv_y"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(ldi.cpu().numpy(), f["maf_inv_ld"], rtol=1e-4, atol=1e-4)
    for use_lu, tag in ((True, "lu"), (False, "w")):
        ia = nf.flows.InvertibleAffine(5, use_lu=use_lu)
        ia.load_state_dict({k[len(f"ia_{tag}__"):]: torch.from_numpy(np.asarray(f[k])) for k in f.files
                            if k.startswith(f"ia_{tag}__")}, strict=True)
        ia = ia.cuda()
        z = cuda(f[f"ia_{tag}_z"])
        a, la = ia.forward(z)
        b, lb = ia.inverse(z)
        np.testing.assert_allclose(a.cpu().numpy(), f[f"ia_{tag}_fwd"], rtol=1e-4, atol=2e-5)
        np.testing.assert_allclose(b.cpu().numpy(), f[f"ia_{tag}_inv"], rtol=1e-4, atol=2e-5)
        assert float(la) == pytest.approx(float(f[f"ia_{tag}_fwd_ld"]), rel=1e-4, abs=1e-5)
        assert float(lb) == pytest.approx(float(f[f"ia_{tag}_inv_ld"]), rel=1e-4, abs=1e-5)


def _residual_model(f, d):
    flows = [nf.flows.Residual(nf.nets.LipschitzMLP([d, 32, 32, d], init_zeros=False, lipschitz_const=0.9), reduce_memory=True)
             for _ in range(3)]
    m = nf.NormalizingFlow(nf.distributions.DiagGaussian(d, trainable=False), flows)
    m.load_state_dict({k[len(f"sd{d}__"):]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith(f"sd{d}__")},
                      strict=True)
    return m.cuda()


@pytest.mark.parametrize("d", [2, 4])
def test_residual_flow_matches_reference(d):
    """SURVEY 8f-3 / BASELINE config 5: Residual(iResBlock(LipschitzMLP)).  Exact 2-D eval path (residual.py:148-161)
    and the power-series estimators with the random truncation and the Hutchinson probe injected (the same values the
    reference was given while tests/golden/make_golden.py residual minted the vectors): eval = basic estimator with 20
    exact terms (:183-192,355-366), training = Neumann surrogate (:368-379)."""
    f = np.load(os.path.join(GOLDEN, "residual.npz"))
    model = _residual_model(f, d)
    x = cuda(f[f"x{d}"])
    n_inj, eps = f[f"n_inj{d}"], f[f"eps{d}"]

    def run(train):
        model.train(train)
        order = list(range(len(model.flows) - 1, -1, -1))  # density pass: last flow first
        for call, i in enumerate(order):
            blk = model.flows[i].iresblock
            blk._inject_n, blk._inject_eps = n_inj[call % 3], cuda(eps[call % 3])
        z, ld = model.inverse_and_log_det(x)
        model.eval()
        return z.cpu().numpy(), ld.cpu().numpy()
    z, ld = run(False)
    np.testing.assert_allclose(z, f[f"eval_z{d}"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(ld, f[f"eval_ld{d}"], rtol=1e-4, atol=5e-5)
    z, ld = run(True)
    np.testing.assert_allclose(z, f[f"train_z{d}"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(ld, f[f"train_ld{d}"], rtol=1e-4, atol=5e-5)
    if d == 2:
        lp = model.log_prob(x).cpu().numpy()
        np.testing.assert_allclose(lp, f["eval_logprob2"], rtol=1e-4, atol=1e-4)
        xs, lds = model.forward_and_log_det(cuda(f["eval_z2"]))   # sampling direction: fixed-point inverse (:130-139)
        np.testing.assert_allclose(xs.cpu().numpy(), f["fwd_x2"], rtol=1e-4, atol=2e-4)
        np.testing.assert_allclose(lds.cpu().numpy(), f["fwd_ld2"], rtol=1e-3, atol=2e-4)
        # unbiasedness of the stochastic estimator: its mean over probes approaches the exact log-det
        blk = model.flows[0].iresblock
        xin = x[:16].repeat(256, 1)
        blk.train(False)
        _, exact = blk._logdetgrad(x[:16])
        torch.manual_seed(0)
        np.random.seed(0)
        acc = torch.zeros(16, device="cuda")
        reps = 24
        for _ in range(reps):
            x4 = torch.cat([xin, torch.zeros(xin.shape[0], 0, device="cuda")], 1)
            blk_est = blk
            blk_est.brute_force = False
            # force the estimator path on 2-D inputs: call it in training mode with basic estimator semantics
            blk_est.training, blk_est.neumann_grad = True, False
            _, est = blk_est._logdetgrad(x4)
            blk_est.training, blk_est.neumann_grad = False, True
            acc += est.view(256, 16).mean(0)
        mean_est = (acc / reps).cpu().numpy()
        assert np.abs(mean_est - exact.view(-1).cpu().numpy()).max() < 0.05, (mean_est, exact.view(-1).cpu().numpy())


def test_conditional_normalizing_flow_with_context():
    """SURVEY 8f-4: ConditionalNormalizingFlow with context-conditioned coupled / autoregressive spline layers (GLU
    context branch) and a ConditionalDiagGaussian base, against the reference (make_golden.py conditional)."""
    f = np.load(os.path.join(GOLDEN, "conditional.npz"))
    torch.manual_seed(51)
    d, c = 6, 3
    flows = []
    for i in range(2):
        flows += [nf.flows.CoupledRationalQuadraticSpline(d, 2, 32, num_context_channels=c, reverse_mask=bool(i % 2))]
        flows += [nf.flows.LULinearPermute(d)]
        flows += [nf.flows.AutoregressiveRationalQuadraticSpline(d, 2, 32, num_context_channels=c)]
    enc = nf.nets.MLP([c, 16, 2 * d])
    model = nf.ConditionalNormalizingFlow(nf.distributions.ConditionalDiagGaussian(d, enc), flows)
    model.load_state_dict({k[4:]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith("sd__")}, strict=True)
    model = model.cuda()
    x, ctx = cuda(f["x"]), cuda(f["context"])
    lp = model.log_prob(x, ctx).cpu().numpy()
    np.testing.assert_allclose(lp, f["log_prob"], rtol=RTOL, atol=ATOL)
    assert float(model.forward_kld(x, ctx)) == pytest.approx(float(f["kld"]), rel=2e-5)
    z, ld = model.inverse_and_log_det(x, ctx)
    np.testing.assert_allclose(z.cpu().numpy(), f["z"], rtol=1e-4, atol=2e-4)
    np.testing.assert_allclose(ld.cpu().numpy(), f["inv_ld"], rtol=1e-4, atol=2e-3)
    xr, ldf = model.forward_and_log_det(cuda(f["z"]), ctx)
    np.testing.assert_allclose(xr.cpu().numpy(), f["fwd_x"], rtol=1e-4, atol=1e-3)
    np.testing.assert_allclose(ldf.cpu().numpy(), f["fwd_ld"], rtol=1e-4, atol=1e-2)
    torch.manual_seed(1)
    xs, lq = model.sample(48, ctx)
    np.testing.assert_allclose(lq.cpu().numpy(), model.log_prob(xs, ctx).cpu().numpy(), rtol=1e-4, atol=2e-2)


def test_class_cond_flow():
    """ClassCondFlow (core.py:368-452): class label to the base only; the layer stack runs as one fused launch."""
    spec, sd, a = load_golden("nsf_coupled_d5_h128_l3")
    inner = build_model(annotate_spec(spec, sd), sd)
    torch.manual_seed(5)
    q0 = nf.distributions.ClassCondDiagGaussian(5, 3)
    with torch.no_grad():
        q0.loc.normal_(0, 0.5)
        q0.log_scale.normal_(0, 0.2)
    model = nf.ClassCondFlow(q0, list(inner.flows)).cuda()
    x = cuda(a["x"])
    y = torch.randint(3, (x.shape[0],), generator=torch.Generator().manual_seed(6)).cuda()
    lp = model.log_prob(x, y).cpu().numpy()
    z, ld = O.inverse_and_log_det(spec, sd, a["x"].astype(np.float64))
    qsd = {"q0.loc": q0.loc.detach().cpu().numpy().astype(np.float64), "q0.log_scale": q0.log_scale.detach().cpu().numpy().astype(np.float64)}
    ref = ld + O.class_cond_diag_gaussian_log_prob(z, y.cpu().numpy(), qsd, "q0.")
    np.testing.assert_allclose(lp, ref, rtol=RTOL, atol=ATOL)
    assert float(model.forward_kld(x, y)) == pytest.approx(-float(ref.mean()), rel=2e-5)
    xs, lq = model.sample(64, y[:64])
    np.testing.assert_allclose(lq.cpu().numpy(), model.log_prob(xs, y[:64]).cpu().numpy(), rtol=1e-4, atol=2e-2)


@pytest.mark.parametrize("cfg", [((6, 256, 256, 12), 16, 16, 7), ((12, 256, 256, 24), 8, 8, 5), ((24, 256, 256, 48), 4, 4, 9)])
def test_glow_conditioner_at_real_width(cfg):
    """ConvNet2d at the real Glow width (hidden 256; examples/glow.ipynb cell 2): the last 3x3 convolution runs as nine
    stacked 1x1 products on the tensor core + a shifted sum (csrc/nfb_glow.cu tap_shift_add_kernel) when 9*cout <= 256,
    as an im2col GEMM otherwise; against the oracle's direct convolution (nets/cnn.py:33-61)."""
    channels, H, W, B = cfg
    torch.manual_seed(sum(channels))
    net = nf.nets.ConvNet2d(channels, (3, 1, 3), leaky=0.0, init_zeros=False).cuda()
    x = torch.randn(B, channels[0], H, W, device="cuda")
    y = net(x).cpu().numpy()
    sd = {"net." + k: v.detach().cpu().numpy().astype(np.float64) for k, v in net.net.state_dict().items()}
    ref = O.convnet2d(x.cpu().numpy().astype(np.float64), sd, "", leaky=0.0)
    scale = np.abs(ref).max()
    assert np.abs(y - ref).max() <= 1e-4 * scale + 1e-5, (np.abs(y - ref).max(), scale)


def test_glow_c3_shape_against_reference_on_this_gpu():
    """BASELINE config 3 at its REAL shape (examples/glow.ipynb cell 2: L=3, K=16, hidden 256, 3x32x32; 48 Glow blocks,
    8 M parameters): the reference's fp64 log_prob (tests/golden/glow_c3.npz, make_golden.py glow_c3) for weights
    rebuilt from seeds plus the stored ActNorm statistics, compared at the stated tolerance (rtol 1e-4 on every row;
    |log_prob| ~ 1e3-1e4 here)."""
    from helpers_glow import build_glow_c3
    f = np.load(os.path.join(GOLDEN, "glow_c3.npz"))
    model, x, y = build_glow_c3(f)
    model = model.cuda()
    lp = model.log_prob(x.cuda(), y.cuda()).cpu().numpy().astype(np.float64)
    rel = np.abs(lp - f["log_prob_f64"]) / np.abs(f["log_prob_f64"])
    print(f"\n[glow C3 shape, 64 images] |log_prob| ~ {np.abs(f['log_prob_f64']).mean():.0f}; rel err max {rel.max():.2e} median {np.median(rel):.2e}")
    assert rel.max() < RTOL, rel.max()


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["cc_s", "cc_t", "ca_s", "ca_t"])
def test_circular_spline_layers_match_reference(tag):
    """SURVEY 8f-4: CircularCoupled / CircularAutoregressive RQ splines (per-feature tails list, periodic features in
    front of the conditioner, scalar and per-feature tail bounds) in both directions against vectors minted from the
    reference (tests/golden/make_golden.py circular); reference checkpoints load strict=True."""
    f = np.load(os.path.join(GOLDEN, "circular.npz"))
    d, tbt = 6, torch.from_numpy(np.asarray(f["tail_bound_tensor"]))
    make = {
        "cc_s": lambda: nf.flows.CircularCoupledRationalQuadraticSpline(d, 2, 32, [0, 2, 5], tail_bound=3.0),
        "cc_t": lambda: nf.flows.CircularCoupledRationalQuadraticSpline(d, 1, 32, [0, 2, 5], tail_bound=tbt.clone(),
                                                                         reverse_mask=True),
        "ca_s": lambda: nf.flows.CircularAutoregressiveRationalQuadraticSpline(d, 2, 32, [1, 3], tail_bound=3.0),
        "ca_t": lambda: nf.flows.CircularAutoregressiveRationalQuadraticSpline(d, 1, 32, [0, 2, 5], tail_bound=tbt.clone(),
                                                                               permute_mask=False),
    }[tag]
    m = make()
    m.load_state_dict({k[len(tag) + 2:]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith(tag + "__")},
                      strict=True)
    m = m.cuda()
    x = cuda(f[f"{tag}_x"])
    y, ld = m.forward(x)
    assert y.shape == x.shape and ld.shape == (x.shape[0],) and ld.dtype == torch.float32
    np.testing.assert_allclose(y.cpu().numpy(), f[f"{tag}_fwd_y"], rtol=1e-4, atol=1e-4)
    # (log-dets: sums over 6 features of log-derivatives of steep splines (weights perturbed by 0.15) whose parameters come
    #  from bf16x3 tensor-core GEMMs, 2^-17 per product: a few 1e-4 absolute on values of order 1)
    np.testing.assert_allclose(ld.cpu().numpy(), f[f"{tag}_fwd_ld"], rtol=1e-4, atol=1e-3)
    xi, ldi = m.inverse(x)
    np.testing.assert_allclose(xi.cpu().numpy(), f[f"{tag}_inv_y"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(ldi.cpu().numpy(), f[f"{tag}_inv_ld"], rtol=1e-4, atol=1e-3)
    # inside a NormalizingFlow (per-layer loop: these layers are not part of the fused stack)
    model = nf.NormalizingFlow(nf.distributions.DiagGaussian(d, trainable=False), [m]).cuda()
    lp = model.log_prob(x)
    ref = f[f"{tag}_inv_ld"] - 0.5 * d * np.log(2 * np.pi) - 0.5 * (f[f"{tag}_inv_y"] ** 2).sum(1)
    np.testing.assert_allclose(lp.cpu().numpy(), ref, rtol=1e-4, atol=1.2e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["plain", "cc"])
def test_glow_base_distribution(tag):
    """GlowBase (distributions/base.py:347-471): log_prob against reference-minted vectors (with / without class
    conditioning and temperature); sample() returns (z, log_p) with log_p == log_prob(z)."""
    f = np.load(os.path.join(GOLDEN, "glow_base.npz"))
    q = nf.distributions.GlowBase((4, 3, 3), num_classes=5 if tag == "cc" else None)
    q.load_state_dict({k[len(tag) + 2:]: torch.from_numpy(np.asarray(f[k])) for k in f.files if k.startswith(tag + "__")},
                      strict=True)
    q = q.cuda()
    z = cuda(f[f"{tag}_z"])
    y = torch.from_numpy(np.asarray(f[f"{tag}_y"])).cuda() if tag == "cc" else None
    lp = q.log_prob(z, y) if tag == "cc" else q.log_prob(z)
    np.testing.assert_allclose(lp.cpu().numpy(), f[f"{tag}_lp"], rtol=1e-5, atol=1e-4)
    q.temperature = 0.7
    lp = q.log_prob(z, y) if tag == "cc" else q.log_prob(z)
    np.testing.assert_allclose(lp.cpu().numpy(), f[f"{tag}_lp_t07"], rtol=1e-5, atol=1e-4)
    q.temperature = None
    zs, lps = q.forward(16, y=y[:16]) if tag == "cc" else q.forward(16)
    assert zs.shape == (16, 4, 3, 3) and lps.shape == (16,)
    again = q.log_prob(zs, y[:16]) if tag == "cc" else q.log_prob(zs)
    np.testing.assert_allclose(lps.cpu().numpy(), again.cpu().numpy(), rtol=1e-6, atol=1e-5)


@pytest.mark.gpu
def test_host_batch_in_flight_repeated_calls():
    """Host-buffer entry points at a batch large enough for the in-flight path (chunked H2D gating the layer-0 tiles of the
    whole-stack kernel): the first call of a batch size enqueues the copies first, repeated calls enqueue the kernels
    first (nfb_api.cu h2d_prepare / h2d_copies) -- every call must reproduce the device-resident result, also when the
    batch size changes in between and for a ragged last tile."""
    import bench
    model = bench.build_model("ar", layers=4).cuda()
    g = torch.Generator().manual_seed(7)
    for rows in (16384 + 37, 16384 + 37, 24576, 16384 + 37, 16384 + 37):
        x = (torch.randn(rows, bench.D, generator=g) * 1.5)
        xh = x.pin_memory()
        ref_lp = model.log_prob(x.cuda()).cpu().numpy()
        ref_kld = float(model.forward_kld(x.cuda()))
        for _ in range(2):
            assert model.forward_kld_host(xh) == pytest.approx(ref_kld, rel=1e-6)
            np.testing.assert_array_equal(model.log_prob_host(xh).numpy(), ref_lp)


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: the last timed step's loss, the last host-entry step's loss and the per-sample log_prob
    of the last timed batch, the same on a second run with the same arguments (seeded inputs and weights)."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    runs = []
    for r in range(2):
        d = tmp_path / f"run{r}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3",
                              "--batch", "8192", "--no-cpu-baseline", "--no-reference-eager", "--no-train-step",
                              "--no-extra-configs", "--dump-outputs", str(d)], capture_output=True, text=True,
                             timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 3
        runs.append({n: np.load(d / f"{n}.npy") for n in ("forward_kld", "forward_kld_host", "log_prob")})
    a, b = runs
    assert a["log_prob"].shape == (8192,) and a["log_prob"].dtype == np.float32 and np.isfinite(a["log_prob"]).all()
    assert float(a["forward_kld"]) == pytest.approx(-float(a["log_prob"].astype(np.float64).mean()), rel=1e-6)
    assert float(b["forward_kld"]) == line["config"]["loss"]
    for n in a:
        np.testing.assert_allclose(a[n], b[n], rtol=1e-6)
