"""Gabor orientation loss (SURVEY.md §8f row 2, first slice): the fused forward/backward kernels of csrc/mg_orient.cu against
the oracle restatement (values and the gradient w.r.t. the image), and the oracle against what the reference's own L1OLoss
class computes on the same inputs (tests/golden/golden_orient_loss.npz)."""
import os

import numpy as np
import pytest
import torch

import michigan_oracle as orc

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_orient_loss.npz")


def _inputs(n=2, size=96, seed=0):
    g = torch.Generator().manual_seed(seed)
    # smooth-ish image so that filter responses have clear winners, plus noise
    yy, xx = torch.meshgrid(torch.arange(size).float(), torch.arange(size).float(), indexing="ij")
    base = torch.sin(0.7 * xx + 0.3 * yy).view(1, 1, size, size) * 0.5
    img = (base + 0.2 * torch.randn(n, 3, size, size, generator=g)).clamp(-1, 1)
    orient = torch.floor(torch.rand(n, 1, size, size, generator=g) * 255)
    sem = torch.zeros(n, 2, size, size)
    sem[:, 1, 10:80, 20:70] = 1
    sem[:, 0] = 1 - sem[:, 1]
    return img, orient, sem


def test_orientation_loss_kernels_vs_oracle():
    from michigan_b200.networks.loss import L1OLoss
    from michigan_b200.options import make_opt
    img, orient, sem = _inputs()
    crit = L1OLoss(make_opt())
    x = img.clone().cuda().requires_grad_()
    lo, lc = crit(x, orient.cuda(), sem.cuda())
    (lo * 10.0 + lc * 100.0).backward()
    xr = img.clone().requires_grad_()
    ro, rc = orc.orient_loss_gabor(xr, orient, sem)
    (ro * 10.0 + rc * 100.0).backward()
    print("orient loss %.6f (oracle %.6f)  confidence loss %.6f (oracle %.6f)" % (float(lo), float(ro), float(lc), float(rc)))
    # the arg-max over 32 responses can tie-break differently for a handful of pixels (fp32 summation order of a 289-tap filter)
    assert abs(float(lo) - float(ro)) <= 2e-4 * max(1.0, abs(float(ro)))
    assert abs(float(lc) - float(rc)) <= 1e-5 * max(1.0, abs(float(rc)))
    g, gr = x.grad.cpu(), xr.grad
    rel = float((g - gr).norm() / gr.norm())
    print("   d/d image: relative L2 error %.3e (|grad| %.3e)" % (rel, float(gr.norm())))
    assert rel <= 2e-2


def test_oracle_orientation_loss_pinned_against_the_reference_class():
    """The reference class's losses and image gradient on _inputs(), recorded by tests/golden/make_golden_orient.py."""
    z = np.load(GOLDEN)
    img = torch.from_numpy(z["img"])
    orient = torch.from_numpy(z["orient"]).float()
    hair = torch.from_numpy(z["hair"]).float()
    sem = torch.cat([1 - hair, hair], 1)
    xr = img.clone().requires_grad_()
    ro, rc = orc.orient_loss_gabor(xr, orient, sem)
    (ro * 10.0 + rc * 100.0).backward()
    g = torch.from_numpy(z["grad"])
    assert abs(float(z["orient_loss"][0]) - float(ro)) <= 2e-4 * max(1.0, abs(float(ro)))
    assert abs(float(z["confidence_loss"][0]) - float(rc)) <= 1e-5 * max(1.0, abs(float(rc)))
    assert float((g - xr.grad).norm() / xr.grad.norm()) <= 2e-2
