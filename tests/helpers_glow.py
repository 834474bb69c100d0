"""Build OUR MultiscaleFlow for the Glow goldens (examples/glow.ipynb cell 2, reduced and real size)."""
import numpy as np
import pytest
import torch

import normflows as nf


def build_glow_small(sd=None, L_=2, K=2, hidden=32, shape=(3, 8, 8), ncls=10):
    q0, merges, flows = [], [], []
    for i in range(L_):
        fl = [nf.flows.GlowBlock(shape[0] * 2 ** (L_ + 1 - i), hidden, split_mode="channel", scale=True)
              for _ in range(K)] + [nf.flows.Squeeze()]
        flows += [fl]
        if i > 0:
            merges += [nf.flows.ImageMerge()]
            ls = (shape[0] * 2 ** (L_ - i), shape[1] // 2 ** (L_ - i), shape[2] // 2 ** (L_ - i))
        else:
            ls = (shape[0] * 2 ** (L_ + 1), shape[1] // 2 ** L_, shape[2] // 2 ** L_)
        q0 += [nf.distributions.ClassCondDiagGaussian(ls, ncls)]
    m = nf.MultiscaleFlow(q0, flows, merges)
    if sd is not None:
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    return m


def build_glow_c3(f):
    """OUR MultiscaleFlow at BASELINE config 3's real shape with the weights of tests/golden/glow_c3.npz, rebuilt by
    the recipe make_golden.py case_glow_c3 describes; every state_dict entry is checked against the stored checksum.
    -> (fp32 model, x, y)."""
    L_, K, hidden, shape, ncls, batch = 3, 16, 256, (3, 32, 32), 10, 64
    torch.manual_seed(0)
    m = build_glow_small(L_=L_, K=K, hidden=hidden, shape=shape, ncls=ncls).double()
    with torch.no_grad():
        gp = torch.Generator().manual_seed(2)
        for _, p in m.named_parameters():
            p.add_(0.02 * torch.randn(p.shape, generator=gp, dtype=torch.float64))
    sd = m.state_dict()
    for k in f.files:
        if k.startswith("sd__"):
            sd[k[4:]] = torch.from_numpy(f[k])
    for k, (s, s2) in zip(f["ck_keys"], f["ck"]):
        v = sd[str(k)].double()
        assert float(v.sum()) == pytest.approx(s, rel=1e-12, abs=1e-12), k
        assert float((v ** 2).sum()) == pytest.approx(s2, rel=1e-12, abs=1e-12), k
    assert len(f["ck_keys"]) == len(sd)
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(batch, *shape, generator=g)
    y = torch.randint(ncls, (batch,), generator=g)
    np.testing.assert_array_equal(x.flatten()[f["x_idx"]].double().numpy(), f["x_sample"])
    np.testing.assert_array_equal(y.numpy(), f["y"])
    return m.float(), x, y
