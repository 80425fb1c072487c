"""Record the reference's Gabor orientation loss (models/networks/loss.py, L1OLoss) on fixed inputs (needs a MichiGAN
checkout, see ref_shims.py):

    python tests/golden/make_golden_orient.py

The reference class places its filter parameters with .cuda(); here Tensor.cuda is the identity, so it runs on the CPU
with its arithmetic unchanged.  golden_orient_loss.npz holds the inputs (image, orientation labels, hair mask), the
two losses and the gradient of 10 * orient_loss + 100 * confidence_loss with respect to the image, which
tests/test_gpu_orient.py compares with the oracle.
"""
import os
import sys
import warnings
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [HERE, os.path.dirname(HERE), ROOT, os.path.join(ROOT, "oracle")]
import ref_shims  # noqa: E402
from test_gpu_orient import _inputs  # noqa: E402


def main():
    ref_shims.import_reference()
    warnings.filterwarnings("ignore")
    torch.Tensor.cuda = lambda self, *a, **k: self
    from models.networks.loss import L1OLoss
    img, orient, sem = _inputs()
    crit = L1OLoss(SimpleNamespace(orient_filter="gabor", use_ig=False))
    x = img.clone().requires_grad_()
    lo, lc = crit(x, orient, sem)
    (lo * 10.0 + lc * 100.0).backward()
    path = os.path.join(HERE, "golden_orient_loss.npz")
    np.savez_compressed(path, img=img.numpy(), orient=orient.numpy().astype(np.uint8), hair=sem[:, 1:2].numpy().astype(np.uint8),
                        orient_loss=np.array([float(lo)]), confidence_loss=np.array([float(lc)]), grad=x.grad.numpy())
    print("orient loss %.6f confidence loss %.6f; wrote %s (%.1f KB)" % (float(lo), float(lc), path, os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
