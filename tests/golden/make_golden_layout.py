"""Record the reference's network layout and seeded initialisation (needs a MichiGAN checkout, see ref_shims.py):

    python tests/golden/make_golden_layout.py

Builds the reference's generator and discriminator (ngf = ndf = 32, 128x128) through its own option parser and
define_G / define_D, and stores in golden_layout_ngf32.npz:
  * layout: every state-dict key in order, with shape and dtype, for G and D;
  * init/<key>: for the generator built right after torch.manual_seed(123), a strided sample of up to 65 values of
    every tensor (float64) and, in init_abs_sum/<key>, the sum of its absolute values over the whole tensor.
tests/test_host_logic.py compares the product's networks with these records.
"""
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shims  # noqa: E402

EXTRA = ["--ngf", "32", "--ndf", "32", "--crop_size", "128", "--load_size", "128"]
INIT_SEED = 123


def init_sample(t):
    f = t.detach().double().reshape(-1)
    return f[::max(1, f.numel() // 64)].numpy()


def main():
    ref_shims.patch_training()
    opt = ref_shims.ref_options(True, EXTRA)
    nets = ref_shims.import_reference()
    with contextlib.redirect_stdout(io.StringIO()):
        refG, refD = nets.define_G(opt), nets.define_D(opt)
    layout = {name: [[k, list(v.shape), str(v.dtype)] for k, v in net.state_dict().items()]
              for name, net in (("G", refG), ("D", refD))}
    out = {"layout": np.frombuffer(json.dumps(layout).encode(), dtype=np.uint8),
           "config": np.frombuffer(json.dumps({"args": EXTRA, "init_seed": INIT_SEED}).encode(), dtype=np.uint8)}
    torch.manual_seed(INIT_SEED)
    with contextlib.redirect_stdout(io.StringIO()):
        refG = nets.define_G(opt)
    for k, v in refG.state_dict().items():
        out["init/" + k] = init_sample(v)
        out["init_abs_sum/" + k] = np.array([v.detach().double().abs().sum().item()])
    path = os.path.join(HERE, "golden_layout_ngf32.npz")
    np.savez_compressed(path, **out)
    print("wrote %s (%.1f KB, %d arrays)" % (path, os.path.getsize(path) / 1024, len(out)))


if __name__ == "__main__":
    main()
