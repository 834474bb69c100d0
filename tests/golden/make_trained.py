"""Mint TRAINED-weight fixtures with the real reference (normflows 1.7.3).

    NFB_REFERENCE=<normalizing-flows checkout> python tests/golden/make_trained.py

The random-perturbation goldens (make_golden.py) have zero-mean, sign-symmetric weights -- the setting the
tensor-core accumulate-truncation compensation (csrc/nfb_kernels.h kAccStepGain) was calibrated on.  Trained
conditioners are different: post-ReLU activations against correlated same-sign weights.  This script trains the
flagship block shape (d=64, hidden 256, 2 blocks, 8 bins) for a few hundred Adam steps with the reference's own
training loop (examples/neural_spline_flow.ipynb cell 4: forward_kld, Adam lr 1e-3... here 5e-4) on a structured
64-d target, then stores PARAMETERS ONLY (masks / degrees / permutations are deterministic functions of the
constructor seed and are rebuilt by the consumer with torch.manual_seed(SEED)) plus fp64 / fp32 reference
outputs for a held-out batch.  Output: tests/golden/trained_<kind>_d64_h256_l4.npz
"""
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.environ["NFB_REFERENCE"])
import normflows as nf  # noqa: E402  (the reference)

HERE = os.path.dirname(os.path.abspath(__file__))
D, LAYERS, HIDDEN, SEED, STEPS, BATCH = 64, 4, 256, 7, 400, 512


def target_sample(n, g):
    """Structured 64-d data: 6 latent factors through a fixed tanh mixing + two-mode offset + small noise."""
    gm = torch.Generator().manual_seed(99)
    A = torch.randn(6, D, generator=gm) * 0.9
    b = torch.randn(D, generator=gm) * 0.5
    u = torch.randn(n, 6, generator=g)
    mode = (torch.rand(n, 1, generator=g) < 0.5).float() * 2 - 1
    return 1.6 * torch.tanh(u @ A + 0.7 * mode * b) + 0.25 * torch.randn(n, D, generator=g)


def build(kind):
    torch.manual_seed(SEED)
    fl = []
    for i in range(LAYERS):
        if kind == "ar":
            fl.append(nf.flows.AutoregressiveRationalQuadraticSpline(D, 2, HIDDEN))
        else:
            fl.append(nf.flows.CoupledRationalQuadraticSpline(D, 2, HIDDEN, reverse_mask=bool(i % 2)))
        fl.append(nf.flows.LULinearPermute(D))
    return nf.NormalizingFlow(nf.distributions.DiagGaussian(D, trainable=False), fl)


def main():
    torch.set_num_threads(os.cpu_count())
    for kind in ("ar", "coupled"):
        model = build(kind)
        g = torch.Generator().manual_seed(1)
        opt = torch.optim.Adam(model.parameters(), lr=5e-4, weight_decay=1e-5)
        t0, hist = time.time(), []
        for it in range(STEPS):
            opt.zero_grad()
            loss = model.forward_kld(target_sample(BATCH, g))
            if not (torch.isnan(loss) | torch.isinf(loss)):
                loss.backward()
                opt.step()
            hist.append(float(loss))
            if it % 50 == 0:
                print(kind, it, f"{float(loss):.3f}", f"{time.time() - t0:.0f}s", flush=True)
        model.eval()
        gx = torch.Generator().manual_seed(2)
        x = torch.cat([target_sample(768, gx), 1.5 * torch.randn(256, D, generator=gx)])  # data + off-manifold rows
        out = {"torch_version": torch.__version__, "x": x.numpy().astype(np.float64),
               "loss_history": np.asarray(hist, dtype=np.float32),
               "meta": json.dumps({"kind": kind, "d": D, "layers": LAYERS, "hidden": HIDDEN, "seed": SEED,
                                   "steps": STEPS, "batch": BATCH})}
        for k, v in model.named_parameters():
            out["sd__" + k] = v.detach().numpy()
        for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
            m = model.to(dt)
            with torch.no_grad():
                out[f"log_prob_{tag}"] = m.log_prob(x.to(dt)).numpy()
                out[f"kld_{tag}"] = m.forward_kld(x.to(dt)).numpy()
        model.to(torch.float32)
        np.savez_compressed(os.path.join(HERE, f"trained_{kind}_d64_h256_l4.npz"), **out)
        rel = np.abs(out["log_prob_f32"] - out["log_prob_f64"]) / np.abs(out["log_prob_f64"])
        print("wrote", kind, "loss", hist[0], "->", hist[-1], "kld", float(out["kld_f64"]),
              "reference fp32-vs-fp64 rel max", rel.max(), flush=True)


if __name__ == "__main__":
    main()
