"""Mint golden vectors from the REAL reference (normflows 1.7.3).

NFB_REFERENCE names the directory that holds the reference's `normflows` package:
    NFB_REFERENCE=<normalizing-flows checkout> python tests/golden/make_golden.py
Writes tests/golden/<case>.npz, each holding:
    spec (json string), sd__<key> (state_dict arrays), x, [y], and for fp64 & fp32:
    log_prob, z, kld, per-layer log_det (ld__<i>) in the density direction, and
    fwd_z / fwd_ld (forward_and_log_det of the latent = sampling direction).
The reference ships no golden vectors (SURVEY.md section 4), so these files are what
pins the oracle (oracle/nf_oracle.py) and the CUDA path to the reference.
torch version used is recorded in each file.
"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.environ["NFB_REFERENCE"])
import normflows as nf  # noqa: E402  (the reference)

HERE = os.path.dirname(os.path.abspath(__file__))


def perturb(model, sigma, seed):
    """Move weights off identity-init (final layer weight 0 hides every bug)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=g, dtype=p.dtype))


def dump(name, model, spec, x, y=None, sampling=True, extra=None):
    out = {"spec": json.dumps(spec), "torch_version": torch.__version__,
           "x": x.numpy().astype(np.float64)}
    if y is not None:
        out["y"] = y.numpy()
    for k, v in model.state_dict().items():
        out["sd__" + k] = v.detach().numpy()  # float32 params are stored exactly; .double() models are casts of these
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        m = model.to(dt)
        xx = x.to(dt)
        with torch.no_grad():
            if spec["kind"] == "MultiscaleFlow":
                lp = m.log_prob(xx, y)
                out[f"log_prob_{tag}"] = lp.numpy()
                out[f"kld_{tag}"] = m.forward_kld(xx, y).numpy()
                # both directions of the multiscale stack (core.py:504-551): latents per level, then back
                zl, ld = m.inverse_and_log_det(xx)
                for j, zj in enumerate(zl):
                    out[f"ms_z{j}_{tag}"] = zj.numpy()
                out[f"ms_inv_ld_{tag}"] = ld.numpy()
                fx, fld = m.forward_and_log_det(zl)
                out[f"ms_fwd_x_{tag}"] = fx.numpy()
                out[f"ms_fwd_ld_{tag}"] = fld.numpy()
                continue
            lp = m.log_prob(xx)
            out[f"log_prob_{tag}"] = lp.numpy()
            out[f"kld_{tag}"] = m.forward_kld(xx).numpy()
            z = xx
            for i in range(len(m.flows) - 1, -1, -1):
                z, ld = m.flows[i].inverse(z)
                out[f"ld_{tag}__{i}"] = (ld * torch.ones(len(xx), dtype=dt)).numpy()
                out[f"zl_{tag}__{i}"] = z.numpy()
            out[f"z_{tag}"] = z.numpy()
            if sampling:
                fz, fld = m.forward_and_log_det(z)
                out[f"fwd_x_{tag}"] = fz.numpy()
                out[f"fwd_ld_{tag}"] = fld.numpy()
    model.to(torch.float32)
    if extra:
        out.update(extra)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("wrote", name, {k: v.shape for k, v in out.items() if k.startswith(("log_prob", "kld"))})


def nsf(kind, d, layers, hidden, blocks, seed, sigma, tail_bound=3.0, bins=8, lu_identity=True):
    torch.manual_seed(seed)
    flows, spec = [], []
    for i in range(layers):
        if kind == "ar":
            flows += [nf.flows.AutoregressiveRationalQuadraticSpline(d, blocks, hidden, num_bins=bins,
                                                                      tail_bound=tail_bound)]
            spec += [{"type": "AutoregressiveRationalQuadraticSpline", "num_input_channels": d,
                      "num_blocks": blocks, "num_hidden_channels": hidden, "num_bins": bins,
                      "tail_bound": tail_bound}]
        else:
            flows += [nf.flows.CoupledRationalQuadraticSpline(d, blocks, hidden, num_bins=bins,
                                                               tail_bound=tail_bound,
                                                               reverse_mask=bool(i % 2))]
            spec += [{"type": "CoupledRationalQuadraticSpline", "num_input_channels": d,
                      "num_blocks": blocks, "num_hidden_channels": hidden, "num_bins": bins,
                      "tail_bound": tail_bound, "reverse_mask": bool(i % 2)}]
        flows += [nf.flows.LULinearPermute(d, identity_init=lu_identity)]
        spec += [{"type": "LULinearPermute", "num_channels": d}]
    q0 = nf.distributions.DiagGaussian(d, trainable=False)
    model = nf.NormalizingFlow(q0, flows)
    perturb(model, sigma, seed + 1)
    return model, {"kind": "NormalizingFlow", "q0": {"type": "DiagGaussian", "shape": [d]},
                   "flows": spec}


def case_spline_edges():
    """Raw spline calls incl. the edge cases of SURVEY 8c.4 (x = +-B exactly, just outside,
    interior-knot hits, |x| >> B, NaN)."""
    from normflows.utils import splines
    torch.manual_seed(7)
    n, k, b = 64, 8, 3.0
    out = {"torch_version": torch.__version__}
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        g = torch.Generator().manual_seed(11)
        uw = torch.randn(n, k, generator=g, dtype=torch.float64).to(dt)
        uh = torch.randn(n, k, generator=g, dtype=torch.float64).to(dt)
        ud = torch.randn(n, k - 1, generator=g, dtype=torch.float64).to(dt)
        x = (torch.randn(n, generator=g, dtype=torch.float64) * 2).to(dt)
        x[0], x[1], x[2], x[3] = b, -b, 3.0000002, -3.0000002
        x[4], x[5], x[6] = 100.0, -1e6, float("nan")
        # interior knot hits: compute knots exactly as the reference does
        w = torch.softmax(uw, -1)
        w = 1e-3 + (1 - 1e-3 * k) * w
        cw = torch.nn.functional.pad(torch.cumsum(w, -1), (1, 0)) * (2 * b) - b
        for j in range(1, 8):
            x[7 + j] = cw[7 + j, j]
        for inv in (False, True):
            y, lad = splines.unconstrained_rational_quadratic_spline(
                x.clone(), uw.clone(), uh.clone(), ud.clone(), inverse=inv, tails="linear",
                tail_bound=b)
            out[f"y_{tag}_{int(inv)}"] = y.numpy()
            out[f"lad_{tag}_{int(inv)}"] = lad.numpy()
        out[f"x_{tag}"], out[f"uw_{tag}"], out[f"uh_{tag}"], out[f"ud_{tag}"] = \
            x.numpy(), uw.numpy(), uh.numpy(), ud.numpy()
    np.savez_compressed(os.path.join(HERE, "spline_edges.npz"), **out)
    print("wrote spline_edges")


def case_realnvp():
    """BASELINE config 1 shape: 8 x [MaskedAffineFlow(MLP[2,4,2] x2), ActNorm(2)] (examples/real_nvp.ipynb)."""
    torch.manual_seed(3)
    flows, spec = [], []
    b = torch.tensor([1.0, 0.0])
    for i in range(8):
        s = nf.nets.MLP([2, 4, 2], init_zeros=True)
        t = nf.nets.MLP([2, 4, 2], init_zeros=True)
        flows += [nf.flows.MaskedAffineFlow(b if i % 2 == 0 else 1 - b, t, s)]
        spec += [{"type": "MaskedAffineFlow"}]
        flows += [nf.flows.ActNorm(2)]
        spec += [{"type": "ActNorm"}]
    model = nf.NormalizingFlow(nf.distributions.DiagGaussian(2), flows)
    x = nf.distributions.TwoMoons().sample(256)
    with torch.no_grad():
        model.log_prob(x)  # ActNorm data-dependent init happens here (flows/normalization.py:33-38)
    perturb(model, 0.2, 4)
    dump("realnvp2d", model, {"kind": "NormalizingFlow", "q0": {"type": "DiagGaussian", "shape": [2]},
                              "flows": spec}, x)


def case_affine_block():
    """README Real NVP: AffineCouplingBlock(MLP[1,64,64,2]) + Permute(2, 'swap')."""
    torch.manual_seed(5)
    flows, spec = [], []
    for i in range(4):
        pm = nf.nets.MLP([1, 64, 64, 2], init_zeros=True)
        flows += [nf.flows.AffineCouplingBlock(pm)]
        spec += [{"type": "AffineCouplingBlock", "net": "mlp", "scale_map": "exp", "split_mode": "channel"}]
        flows += [nf.flows.Permute(2, mode="swap")]
        spec += [{"type": "Permute", "mode": "swap"}]
    model = nf.NormalizingFlow(nf.distributions.DiagGaussian(2), flows)
    perturb(model, 0.1, 6)
    x = torch.randn(128, 2, generator=torch.Generator().manual_seed(8))
    dump("affine_block2d", model, {"kind": "NormalizingFlow", "q0": {"type": "DiagGaussian", "shape": [2]},
                                   "flows": spec}, x)
    # 6-D variant with shuffle permute and odd split sizes
    torch.manual_seed(9)
    flows, spec = [], []
    for i in range(3):
        pm = nf.nets.MLP([3, 32, 32, 6], init_zeros=False)
        mode = "channel" if i % 2 == 0 else "channel_inv"
        flows += [nf.flows.AffineCouplingBlock(pm, scale_map=["exp", "sigmoid", "sigmoid_inv"][i],
                                               split_mode=mode)]
        spec += [{"type": "AffineCouplingBlock", "net": "mlp",
                  "scale_map": ["exp", "sigmoid", "sigmoid_inv"][i], "split_mode": mode}]
        flows += [nf.flows.Permute(6, mode="shuffle")]
        spec += [{"type": "Permute", "mode": "shuffle"}]
    model = nf.NormalizingFlow(nf.distributions.DiagGaussian(6), flows)
    perturb(model, 0.05, 10)
    x = torch.randn(96, 6, generator=torch.Generator().manual_seed(12))
    dump("affine_block6d", model, {"kind": "NormalizingFlow", "q0": {"type": "DiagGaussian", "shape": [6]},
                                   "flows": spec}, x)


def case_glow():
    """examples/glow.ipynb cell 2 at reduced size: L=2, K=2, hidden 32, 3x8x8, 10 classes."""
    torch.manual_seed(13)
    L, K, hidden, shape, ncls = 2, 2, 32, (3, 8, 8), 10
    q0, merges, flows, levels = [], [], [], []
    for i in range(L):
        flows_, lv = [], []
        for j in range(K):
            c = shape[0] * 2 ** (L + 1 - i)
            flows_ += [nf.flows.GlowBlock(c, hidden, split_mode="channel", scale=True)]
            lv += [{"type": "GlowBlock", "channels": c, "hidden_channels": hidden}]
        flows_ += [nf.flows.Squeeze()]
        lv += [{"type": "Squeeze"}]
        flows += [flows_]
        levels += [lv]
        if i > 0:
            merges += [nf.flows.Merge()]
            ls = (shape[0] * 2 ** (L - i), shape[1] // 2 ** (L - i), shape[2] // 2 ** (L - i))
        else:
            ls = (shape[0] * 2 ** (L + 1), shape[1] // 2 ** L, shape[2] // 2 ** L)
        q0 += [nf.distributions.ClassCondDiagGaussian(ls, ncls)]
    model = nf.MultiscaleFlow(q0, flows, merges)
    g = torch.Generator().manual_seed(14)
    x = torch.rand(16, *shape, generator=g)
    y = torch.randint(ncls, (16,), generator=g)
    with torch.no_grad():
        model.log_prob(x, y)  # ActNorm init
    perturb(model, 0.03, 15)
    dump("glow_small", model, {"kind": "MultiscaleFlow", "levels": levels, "class_cond": True,
                               "num_classes": ncls}, x, y)
    # ActNorm data-dependent init statistics, on their own
    an = nf.flows.ActNorm((6, 1, 1))
    xx = torch.randn(8, 6, 4, 4, generator=g).double() * 2 + 0.5
    an = an.double()
    with torch.no_grad():
        zz, ld = an.inverse(xx)
    np.savez_compressed(os.path.join(HERE, "actnorm_init.npz"), x=xx.numpy(), s=an.s.detach().numpy(),
                        t=an.t.detach().numpy(), z=zz.numpy(), ld=ld.numpy())
    print("wrote actnorm_init")


def main():
    case_spline_edges()
    # the survey's sanity anchors (SURVEY.md 8c.2) are re-derived by tests from these files
    for kind in ("ar", "coupled"):
        m, spec = nsf(kind, 64, 2, 256, 2, seed=0, sigma=0.05)
        x = torch.randn(48, 64, generator=torch.Generator().manual_seed(1234)) * 1.5
        dump(f"nsf_{kind}_d64_h256_l2", m, spec, x, sampling=(kind == "coupled"))
        m, spec = nsf(kind, 5, 3, 128, 2, seed=20, sigma=0.1, lu_identity=False)
        x = torch.randn(64, 5, generator=torch.Generator().manual_seed(21)) * 1.5
        dump(f"nsf_{kind}_d5_h128_l3", m, spec, x)
        m, spec = nsf(kind, 2, 2, 32, 1, seed=30, sigma=0.2, tail_bound=2.0, bins=4, lu_identity=False)
        x = torch.randn(64, 2, generator=torch.Generator().manual_seed(31)) * 1.5
        dump(f"nsf_{kind}_d2_h32_l2_k4", m, spec, x)
    case_realnvp()
    case_affine_block()
    case_glow()


if __name__ == "__main__" and len(sys.argv) == 1:
    main()
if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "glow":
    case_glow()


def case_spline_grads():
    """Gradients of the reference's spline element op w.r.t. every input, by its own autograd in fp64
    (utils/splines.py:16-97, forward branch): loss = sum(cy * y + cl * logabsdet) with random per-element
    weights, so the fixture pins d y / d . and d logabsdet / d . separately for each element."""
    from normflows.utils.splines import unconstrained_rational_quadratic_spline as urqs
    g = torch.Generator().manual_seed(77)
    n, K = 600, 8
    x = (torch.randn(n, generator=g, dtype=torch.float64) * 2.2).requires_grad_(True)  # ~17 % in the tails
    uw = (torch.randn(n, K, generator=g, dtype=torch.float64) * 1.5).requires_grad_(True)
    uh = (torch.randn(n, K, generator=g, dtype=torch.float64) * 1.5).requires_grad_(True)
    ud = (torch.randn(n, K - 1, generator=g, dtype=torch.float64) * 1.5).requires_grad_(True)
    cy = torch.randn(n, generator=g, dtype=torch.float64)
    cl = torch.randn(n, generator=g, dtype=torch.float64)
    y, lad = urqs(x, uw, uh, ud, inverse=False, tail_bound=3.0)
    (cy * y + cl * lad).sum().backward()
    np.savez_compressed(os.path.join(HERE, "spline_grads.npz"), x=x.detach().numpy(), uw=uw.detach().numpy(),
                        uh=uh.detach().numpy(), ud=ud.detach().numpy(), cy=cy.numpy(), cl=cl.numpy(),
                        y=y.detach().numpy(), lad=lad.detach().numpy(), gx=x.grad.numpy(), guw=uw.grad.numpy(),
                        guh=uh.grad.numpy(), gud=ud.grad.numpy(), torch_version=torch.__version__)
    print("wrote spline_grads")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "spline_grads":
    case_spline_grads()


def case_grads():
    """Gradients of forward_kld w.r.t. every parameter and the input (fp64), for the autograd check."""
    for kind in ("ar", "coupled"):
        m, spec = nsf(kind, 5, 3, 128, 2, seed=20, sigma=0.1, lu_identity=False)
        m = m.double()
        x = (torch.randn(64, 5, generator=torch.Generator().manual_seed(21)) * 1.5).double().requires_grad_(True)
        loss = m.forward_kld(x)
        loss.backward()
        out = {"x": x.detach().numpy(), "kld": loss.detach().numpy(), "grad__x": x.grad.numpy()}
        for k, p in m.named_parameters():
            if p.grad is not None:
                out["grad__" + k] = p.grad.numpy()
        np.savez_compressed(os.path.join(HERE, f"grads_nsf_{kind}_d5_h128_l3.npz"), **out)
        print("wrote grads", kind, len(out))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "grads":
    case_grads()


def case_ar64_sampling():
    """Sampling direction of the flagship autoregressive shape (d=64, hidden 256): D = 64 sequential conditioner
    passes per layer (flows/affine/autoregressive.py:29-38).  Same model as nsf_ar_d64_h256_l2 (same constructor
    seed and perturbation), latents = that fixture's z; stores only the sampling-direction outputs (small file).
        python tests/golden/make_golden.py ar64fwd"""
    m, spec = nsf("ar", 64, 2, 256, 2, seed=0, sigma=0.05)
    x = torch.randn(48, 64, generator=torch.Generator().manual_seed(1234)) * 1.5
    out = {"torch_version": torch.__version__}
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        mm = m.to(dt)
        with torch.no_grad():
            z, _ = mm.inverse_and_log_det(x.to(dt))
            fx, fld = mm.forward_and_log_det(z)
            out[f"z_{tag}"], out[f"fwd_x_{tag}"], out[f"fwd_ld_{tag}"] = z.numpy(), fx.numpy(), fld.numpy()
            # one layer alone (flows.0 = autoregressive block) on the latents
            y0, ld0 = mm.flows[0].forward(z)
            out[f"l0_fwd_x_{tag}"], out[f"l0_fwd_ld_{tag}"] = y0.numpy(), ld0.numpy()
    m.to(torch.float32)
    np.savez_compressed(os.path.join(HERE, "nsf_ar_d64_h256_l2_fwd.npz"), **out)
    print("wrote nsf_ar_d64_h256_l2_fwd; round trip err", np.abs(out["fwd_x_f64"] - x.numpy()).max(),
          "f32 spread", np.abs(out["fwd_x_f32"] - out["fwd_x_f64"]).max())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "ar64fwd":
    case_ar64_sampling()


def case_grads_d64():
    """Gradients of forward_kld at the flagship block shape (d=64, hidden 256, 2 blocks; same models and inputs as
    nsf_{ar,coupled}_d64_h256_l2), fp64 autograd of the reference.  Small tensors are stored whole; weight matrices as
    two seeded random projections (grad @ v, u @ grad), which pin every entry without storing 5 MB per model.
        python tests/golden/make_golden.py grads64"""
    for kind in ("ar", "coupled"):
        m, spec = nsf(kind, 64, 2, 256, 2, seed=0, sigma=0.05)
        m = m.double()
        x = (torch.randn(48, 64, generator=torch.Generator().manual_seed(1234)) * 1.5).double().requires_grad_(True)
        loss = m.forward_kld(x)
        loss.backward()
        out = {"x": x.detach().numpy(), "kld": loss.detach().numpy(), "grad__x": x.grad.numpy()}
        g = torch.Generator().manual_seed(77)
        for k, p in m.named_parameters():
            if p.grad is None:
                continue
            if p.grad.numel() <= 4096 or p.grad.dim() != 2:
                out["grad__" + k] = p.grad.numpy()
            else:
                v = torch.randn(p.shape[1], generator=g, dtype=torch.float64)
                u = torch.randn(p.shape[0], generator=g, dtype=torch.float64)
                out["gradv__" + k], out["gradu__" + k] = (p.grad @ v).numpy(), (u @ p.grad).numpy()
                out["projv__" + k], out["proju__" + k] = v.numpy(), u.numpy()
                out["gnorm__" + k] = np.asarray(p.grad.norm().item())
        np.savez_compressed(os.path.join(HERE, f"grads_nsf_{kind}_d64_h256_l2.npz"), **out)
        print("wrote grads64", kind, len(out), float(loss))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "grads64":
    case_grads_d64()


def case_options():
    """Reference options the round-1 shims rejected (VERDICT r1 missing #7): GlowBlock with the plain-matrix
    Invertible1x1Conv (use_lu=False, mixing.py:85-86,110-117,126-129) and ActNorm inside the conditioner
    (net_actnorm=True, nets/cnn.py:45-46), MultiscaleFlow(transform=Logit) (transforms.py:8-47), temperature-annealed
    base distributions, and stand-alone calls of nets.MLP / ResidualNet / MADE.
        python tests/golden/make_golden.py options"""
    torch.manual_seed(21)
    L, K, hidden, shape, ncls = 2, 2, 16, (3, 8, 8), 10
    q0, merges, flows = [], [], []
    for i in range(L):
        flows_ = []
        for j in range(K):
            c = shape[0] * 2 ** (L + 1 - i)
            flows_ += [nf.flows.GlowBlock(c, hidden, split_mode="channel", scale=True, use_lu=False, net_actnorm=True)]
        flows_ += [nf.flows.Squeeze()]
        flows += [flows_]
        if i > 0:
            merges += [nf.flows.Merge()]
            ls = (shape[0] * 2 ** (L - i), shape[1] // 2 ** (L - i), shape[2] // 2 ** (L - i))
        else:
            ls = (shape[0] * 2 ** (L + 1), shape[1] // 2 ** L, shape[2] // 2 ** L)
        q0 += [nf.distributions.ClassCondDiagGaussian(ls, ncls)]
    model = nf.MultiscaleFlow(q0, flows, merges, transform=nf.transforms.Logit(0.05))
    g = torch.Generator().manual_seed(22)
    x = torch.rand(16, *shape, generator=g)
    y = torch.randint(ncls, (16,), generator=g)
    with torch.no_grad():
        model.log_prob(x, y)  # every ActNorm (flow-level and inside the conditioners) initialises here
    perturb(model, 0.03, 23)
    out = {"torch_version": torch.__version__, "x": x.numpy().astype(np.float64), "y": y.numpy()}
    for k, v in model.state_dict().items():
        out["sd__" + k] = v.detach().numpy()
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        m = model.to(dt)
        with torch.no_grad():
            out[f"log_prob_{tag}"] = m.log_prob(x.to(dt), y).numpy()
            for q in m.q0:
                q.temperature = 0.7
            out[f"log_prob_T07_{tag}"] = m.log_prob(x.to(dt), y).numpy()
            for q in m.q0:
                q.temperature = None
            zl, ld = m.inverse_and_log_det(x.to(dt))
            fx, fld = m.forward_and_log_det(zl)
            out[f"inv_ld_{tag}"], out[f"fwd_x_{tag}"], out[f"fwd_ld_{tag}"] = ld.numpy(), fx.numpy(), fld.numpy()
            for j, zj in enumerate(zl):
                out[f"z{j}_{tag}"] = zj.numpy()
    model.to(torch.float32)
    # stand-alone conditioner modules
    torch.manual_seed(24)
    nets = {"mlp": nf.nets.MLP([5, 16, 16, 3], leaky=0.1), "mlp_relu": nf.nets.MLP([5, 16, 3]),
            "resnet": nf.nets.ResidualNet(5, 7, 32, num_blocks=2), "made": nf.nets.MADE(5, 32, output_multiplier=3)}
    xin = torch.randn(33, 5, generator=g)
    out["net_x"] = xin.numpy()
    for name, net in nets.items():
        perturb(net, 0.1, 25)
        for k, v in net.state_dict().items():
            out[f"net__{name}__{k}"] = v.detach().numpy()
        with torch.no_grad():
            out[f"net_y__{name}"] = net.double()(xin.double()).numpy()
    np.savez_compressed(os.path.join(HERE, "options.npz"), **out)
    print("wrote options", out["log_prob_f64"][:3], np.abs(out["fwd_x_f64"] - out["x"]).max())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "options":
    case_options()


def case_neighbours():
    """SURVEY 8f-4 neighbouring layers: MaskedAffineAutoregressive (flows/affine/autoregressive.py:50-128) and
    InvertibleAffine (flows/mixing.py:136-207), per-layer vectors in both directions.
        python tests/golden/make_golden.py neighbours"""
    torch.manual_seed(31)
    g = torch.Generator().manual_seed(32)
    out = {"torch_version": torch.__version__}
    maf = nf.flows.MaskedAffineAutoregressive(6, 32, num_blocks=2)
    perturb(maf, 0.1, 33)
    x = torch.randn(40, 6, generator=g)
    out["maf_x"] = x.numpy()
    for k, v in maf.state_dict().items():
        out["maf__" + k] = v.detach().numpy()
    md = maf.double()
    with torch.no_grad():
        y, ld = md.forward(x.double())
        xi, ldi = md.inverse(x.double())
    out["maf_fwd_y"], out["maf_fwd_ld"], out["maf_inv_y"], out["maf_inv_ld"] = y.numpy(), ld.numpy(), xi.numpy(), ldi.numpy()
    for use_lu in (True, False):
        ia = nf.flows.InvertibleAffine(5, use_lu=use_lu)
        perturb(ia, 0.05, 34)
        tag = "lu" if use_lu else "w"
        z = torch.randn(24, 5, generator=g)
        out[f"ia_{tag}_z"] = z.numpy()
        for k, v in ia.state_dict().items():
            out[f"ia_{tag}__" + k] = v.detach().numpy()
        iad = ia.double()
        with torch.no_grad():
            f, lf = iad.forward(z.double())
            b, lb = iad.inverse(z.double())
        out[f"ia_{tag}_fwd"], out[f"ia_{tag}_fwd_ld"], out[f"ia_{tag}_inv"], out[f"ia_{tag}_inv_ld"] = \
            f.numpy(), np.asarray(lf.numpy()), b.numpy(), np.asarray(lb.numpy())
    np.savez_compressed(os.path.join(HERE, "neighbours.npz"), **out)
    print("wrote neighbours")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "neighbours":
    case_neighbours()


def case_residual():
    """BASELINE config 5 family: Residual (iResBlock) with a LipschitzMLP (flows/residual.py, nets/lipschitz.py).
    Exact 2-D eval path (deterministic), and the stochastic power-series estimators with the random truncation n and
    the Hutchinson probe INJECTED (np.random.geometric / torch.randn_like patched while minting) so that the values
    are reproducible: eval-mode basic estimator (4-D) and training-mode Neumann surrogate (2-D and 4-D).
        python tests/golden/make_golden.py residual"""
    from normflows.flows import residual as R
    torch.manual_seed(41)
    g = torch.Generator().manual_seed(42)
    out = {"torch_version": torch.__version__}
    for d in (2, 4):
        flows = []
        for _ in range(3):
            net = nf.nets.LipschitzMLP([d, 32, 32, d], init_zeros=False, lipschitz_const=0.9)
            flows += [nf.flows.Residual(net, reduce_memory=True)]
        model = nf.NormalizingFlow(nf.distributions.DiagGaussian(d, trainable=False), flows)
        perturb(model, 0.4, 43 + d)
        with torch.no_grad():
            nf.utils.update_lipschitz(model, 50)
        x = torch.randn(64, d, generator=g) * 1.2
        out[f"x{d}"] = x.numpy()
        for k, v in model.state_dict().items():
            out[f"sd{d}__" + k] = v.detach().numpy()
        md = model.double()
        n_inj = [np.array([3]), np.array([1]), np.array([2])]          # one draw per block, in call order
        eps = torch.randn(3, 64, d, generator=g, dtype=torch.float64)
        out[f"n_inj{d}"], out[f"eps{d}"] = np.stack(n_inj), eps.numpy()

        def run(train):
            calls = {"i": 0, "j": 0}
            orig_geo, orig_rl = np.random.geometric, torch.randn_like

            def geo(p, n):
                i = calls["i"]; calls["i"] += 1
                return n_inj[i % 3]

            def rl(t, **kw):
                j = calls["j"]; calls["j"] += 1
                return eps[j % 3].to(t)
            np.random.geometric, torch.randn_like = geo, rl
            try:
                md.train(train)
                # density pass applies flows last-to-first: block 2 is called first -> inject in that order
                z, ld = md.inverse_and_log_det(x.double())
                return z.detach().numpy(), ld.detach().numpy()
            finally:
                np.random.geometric, torch.randn_like = orig_geo, orig_rl
                md.eval()
        z, ld = run(False)
        out[f"eval_z{d}"], out[f"eval_ld{d}"] = z, ld
        z, ld = run(True)
        out[f"train_z{d}"], out[f"train_ld{d}"] = z, ld
        if d == 2:
            with torch.no_grad():
                out["eval_logprob2"] = md.log_prob(x.double()).numpy()
                xs, lds = md.forward_and_log_det(torch.from_numpy(out["eval_z2"]))
            out["fwd_x2"], out["fwd_ld2"] = xs.detach().numpy(), lds.detach().numpy()
    np.savez_compressed(os.path.join(HERE, "residual.npz"), **out)
    print("wrote residual", out["eval_ld2"][:3], out["train_ld2"][:3], np.abs(out["fwd_x2"] - out["x2"]).max())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "residual":
    case_residual()


def case_conditional():
    """ConditionalNormalizingFlow (core.py:216-366) with context-conditioned spline layers (GLU context branch of
    nets/resnet.py:48-50 and nets/made.py:212-214, context layers :261-262,:297-300) and ConditionalDiagGaussian.
        python tests/golden/make_golden.py conditional"""
    torch.manual_seed(51)
    d, c = 6, 3
    flows = []
    for i in range(2):
        flows += [nf.flows.CoupledRationalQuadraticSpline(d, 2, 32, num_context_channels=c, reverse_mask=bool(i % 2))]
        flows += [nf.flows.LULinearPermute(d)]
        flows += [nf.flows.AutoregressiveRationalQuadraticSpline(d, 2, 32, num_context_channels=c)]
    enc = nf.nets.MLP([c, 16, 2 * d])
    model = nf.ConditionalNormalizingFlow(nf.distributions.base.ConditionalDiagGaussian(d, enc), flows)
    perturb(model, 0.1, 52)
    g = torch.Generator().manual_seed(53)
    x = torch.randn(48, d, generator=g) * 1.3
    ctx = torch.randn(48, c, generator=g)
    out = {"torch_version": torch.__version__, "x": x.numpy(), "context": ctx.numpy()}
    for k, v in model.state_dict().items():
        out["sd__" + k] = v.detach().numpy()
    md = model.double()
    with torch.no_grad():
        out["log_prob"] = md.log_prob(x.double(), ctx.double()).numpy()
        out["kld"] = md.forward_kld(x.double(), ctx.double()).numpy()
        z, ld = md.inverse_and_log_det(x.double(), ctx.double())
        xr, ldf = md.forward_and_log_det(z, ctx.double())
    out["z"], out["inv_ld"], out["fwd_x"], out["fwd_ld"] = z.numpy(), ld.numpy(), xr.numpy(), ldf.numpy()
    np.savez_compressed(os.path.join(HERE, "conditional.npz"), **out)
    print("wrote conditional", out["log_prob"][:3], np.abs(out["fwd_x"] - out["x"]).max())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "conditional":
    case_conditional()


def case_circular():
    """SURVEY 8f-4: circular NSF layers (flows/neural_spline/wrapper.py:88-183, 247-311): per-feature tails list, periodic
    features in front of the conditioner, scalar AND per-feature tail bounds; per-layer vectors in both directions.
        python tests/golden/make_golden.py circular"""
    torch.manual_seed(41)
    g = torch.Generator().manual_seed(42)
    out = {"torch_version": torch.__version__}
    d = 6
    tbt = torch.tensor([np.pi, 2.0, np.pi, 4.0, 3.0, np.pi])
    cases = {
        "cc_s": lambda: nf.flows.CircularCoupledRationalQuadraticSpline(d, 2, 32, [0, 2, 5], tail_bound=3.0),
        "cc_t": lambda: nf.flows.CircularCoupledRationalQuadraticSpline(d, 1, 32, [0, 2, 5], tail_bound=tbt.clone(),
                                                                         reverse_mask=True),
        "ca_s": lambda: nf.flows.CircularAutoregressiveRationalQuadraticSpline(d, 2, 32, [1, 3], tail_bound=3.0),
        "ca_t": lambda: nf.flows.CircularAutoregressiveRationalQuadraticSpline(d, 1, 32, [0, 2, 5], tail_bound=tbt.clone(),
                                                                               permute_mask=False),
    }
    for tag, make in cases.items():
        m = make()
        perturb(m, 0.15, 43)
        x = torch.randn(48, d, generator=g) * 1.6   # some coordinates beyond the smaller bounds -> identity branch
        out[f"{tag}_x"] = x.numpy()
        for k, v in m.state_dict().items():
            out[f"{tag}__" + k] = v.detach().numpy()
        md = m.double()
        with torch.no_grad():
            y, ld = md.forward(x.double())
            xi, ldi = md.inverse(x.double())
        out[f"{tag}_fwd_y"], out[f"{tag}_fwd_ld"] = y.numpy(), ld.numpy()
        out[f"{tag}_inv_y"], out[f"{tag}_inv_ld"] = xi.numpy(), ldi.numpy()
    out["tail_bound_tensor"] = tbt.numpy()
    np.savez_compressed(os.path.join(HERE, "circular.npz"), **out)
    print("wrote circular")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "circular":
    case_circular()


def case_glow_base():
    """GlowBase (distributions/base.py:347-471): per-channel Gaussian, with and without class conditioning, with and
    without temperature; log_prob in fp64.    python tests/golden/make_golden.py glow_base"""
    g = torch.Generator().manual_seed(52)
    out = {"torch_version": torch.__version__}
    for tag, ncls in (("plain", None), ("cc", 5)):
        torch.manual_seed(51)
        q = nf.distributions.GlowBase((4, 3, 3), num_classes=ncls)
        perturb(q, 0.3, 53)
        z = torch.randn(20, 4, 3, 3, generator=g) * 1.3
        y = torch.randint(5, (20,), generator=g) if ncls else None
        out[f"{tag}_z"] = z.numpy()
        if y is not None:
            out[f"{tag}_y"] = y.numpy()
        for k, v in q.state_dict().items():
            out[f"{tag}__" + k] = v.detach().numpy()
        qd = q.double()
        with torch.no_grad():
            out[f"{tag}_lp"] = (qd.log_prob(z.double(), y) if ncls else qd.log_prob(z.double())).numpy()
            qd.temperature = 0.7
            out[f"{tag}_lp_t07"] = (qd.log_prob(z.double(), y) if ncls else qd.log_prob(z.double())).numpy()
    np.savez_compressed(os.path.join(HERE, "glow_base.npz"), **out)
    print("wrote glow_base")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "glow_base":
    case_glow_base()


def case_spline_circular():
    """utils/splines.py:42-47 tails="circular" (K derivative parameters, knot K repeats knot 0; identity outside):
    element-wise vectors for the nd = K mode of nfb_rqs_spline_tails.    python tests/golden/make_golden.py spline_circular"""
    from normflows.utils import splines
    g = torch.Generator().manual_seed(61)
    n, K = 500, 8
    x = torch.randn(n, generator=g, dtype=torch.float64) * 2.2
    uw = torch.randn(n, K, generator=g, dtype=torch.float64) * 1.5
    uh = torch.randn(n, K, generator=g, dtype=torch.float64) * 1.5
    ud = torch.randn(n, K, generator=g, dtype=torch.float64) * 1.5
    out = {"torch_version": torch.__version__, "x": x.numpy(), "uw": uw.numpy(), "uh": uh.numpy(), "ud": ud.numpy()}
    for inv in (0, 1):
        y, lad = splines.unconstrained_rational_quadratic_spline(x, uw.clone(), uh.clone(), ud.clone(), inverse=bool(inv),
                                                                 tails="circular", tail_bound=3.0)
        out[f"y_{inv}"], out[f"lad_{inv}"] = y.numpy(), lad.numpy()
    np.savez_compressed(os.path.join(HERE, "spline_circular.npz"), **out)
    print("wrote spline_circular")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "spline_circular":
    case_spline_circular()


def case_glow_c3():
    """BASELINE config 3 at its real shape (examples/glow.ipynb cell 2: L=3, K=16, hidden 256, 3x32x32, 10 classes;
    48 Glow blocks, 8 M parameters), log_prob in fp64.  The weights are too large to store, so most of them are
    rebuilt from seeds by the consumer (tests/helpers_glow.py build_glow_c3): the constructor runs under
    torch.manual_seed(0) in fp32, the model is cast to fp64, and every parameter, in model.parameters() order, gets
    0.02 * randn from a Generator seeded with 2; the inputs are torch.rand / torch.randint from a Generator seeded
    with 1.  Stored: the entries that recipe does not reproduce (the data-dependent ActNorm statistics), a
    (sum, sum of squares) checksum of every state_dict entry, a seeded sample of the inputs, and log_prob.
        python tests/golden/make_golden.py glow_c3"""
    L, K, hidden, shape, ncls, batch = 3, 16, 256, (3, 32, 32), 10, 64
    torch.manual_seed(0)
    q0, merges, flows = [], [], []
    for i in range(L):
        flows_ = [nf.flows.GlowBlock(shape[0] * 2 ** (L + 1 - i), hidden, split_mode="channel", scale=True)
                  for _ in range(K)]
        flows += [flows_ + [nf.flows.Squeeze()]]
        if i > 0:
            merges += [nf.flows.Merge()]
            ls = (shape[0] * 2 ** (L - i), shape[1] // 2 ** (L - i), shape[2] // 2 ** (L - i))
        else:
            ls = (shape[0] * 2 ** (L + 1), shape[1] // 2 ** L, shape[2] // 2 ** L)
        q0 += [nf.distributions.ClassCondDiagGaussian(ls, ncls)]
    model = nf.MultiscaleFlow(q0, flows, merges).double()
    seeded = {k: v.detach().clone() for k, v in model.state_dict().items()}
    g = torch.Generator().manual_seed(1)
    x = torch.rand(batch, *shape, generator=g).double()
    y = torch.randint(ncls, (batch,), generator=g)
    with torch.no_grad():
        model.log_prob(x, y)  # ActNorm data-dependent init
        gp = torch.Generator().manual_seed(2)
        for k, p in model.named_parameters():  # move the zero-initialised last convolutions / base off their init
            d = 0.02 * torch.randn(p.shape, generator=gp, dtype=torch.float64)
            p.add_(d)
            seeded[k] += d
        lp = model.log_prob(x, y)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    keys = sorted(sd)
    idx = np.random.default_rng(0).choice(x.numel(), 512, replace=False)
    out = {"torch_version": torch.__version__, "log_prob_f64": lp.numpy(), "y": y.numpy(), "x_idx": idx,
           "x_sample": x.flatten()[idx].numpy(), "ck_keys": np.array(keys),
           "ck": np.array([[float(sd[k].double().sum()), float((sd[k].double() ** 2).sum())] for k in keys])}
    for k in keys:
        if not torch.equal(sd[k], seeded[k]):
            out["sd__" + k] = sd[k].numpy()
    np.savez_compressed(os.path.join(HERE, "glow_c3.npz"), **out)
    print("wrote glow_c3:", sum(k.startswith("sd__") for k in out), "stored entries of", len(keys), "; log_prob",
          lp[:3].numpy())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "glow_c3":
    case_glow_c3()
