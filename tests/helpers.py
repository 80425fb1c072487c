"""Shared test helpers: golden fixture access, oracle state construction, comparison utilities."""
import json
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = [os.path.join(HERE, "golden", f) for f in ("golden_ngf64_128.npz", "golden_ngf64_128_state.npz")]


class _Golden(dict):
    """The arrays of all GOLDEN files; `files` lists their names as np.load's result does."""

    @property
    def files(self):
        return list(self)


def load_golden():
    z = _Golden()
    for path in GOLDEN:
        with np.load(path) as f:
            z.update({k: f[k] for k in f.files})
    cfg = json.loads(bytes(z["config"]).decode())
    return z, cfg


def summary(t, stride=37, cap=4096):
    f = t.detach().float().cpu().reshape(-1)
    return np.concatenate([np.array([f.mean().item(), f.std().item(), f.abs().max().item(), f.abs().mean().item()],
                                    dtype=np.float64).astype(np.float32), f[::stride][:cap].numpy()])


def assert_summary_close(name, got_t, ref_summary, rel, stride=37):
    """Compare a tensor with a stored (stats + strided subsample) summary, relative to its abs-max."""
    got = summary(got_t, stride)
    scale = max(float(ref_summary[2]), 1e-6)
    err_stats = np.abs(got[:4] - ref_summary[:4]).max()
    err_samp = np.abs(got[4:] - ref_summary[4:]).max() if got.shape == ref_summary.shape else np.inf
    assert got.shape == ref_summary.shape, "%s: shape %s vs %s" % (name, got.shape, ref_summary.shape)
    assert err_samp <= rel * scale and err_stats <= rel * scale, \
        "%s: sample err %.3e stats err %.3e (scale %.3e, rel tol %g)" % (name, err_samp, err_stats, scale, rel)
    return err_samp / scale


def reference_layout_state(kind, cfg, seed):
    """A CPU state dict with the reference's key layout, filled by the deterministic recipe.  The layout
    comes from the product's own (CPU-constructible) module classes, whose keys/shapes are asserted to
    equal the reference's in tests/test_host_logic.py."""
    from michigan_b200 import networks
    from michigan_b200.options import make_opt
    from michigan_b200.synth import fill_state_dict
    opt = make_opt(ngf=cfg["ngf"], ndf=cfg["ndf"], crop_size=cfg["size"], gpu_ids=[])
    net = networks.SPADEBGenerator(opt) if kind == "G" else networks.MultiscaleDiscriminator(opt)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    fill_state_dict(sd, seed)
    return sd


def preprocessed(cfg, n=None, size=None, seed=None):
    """synthetic_batch -> the tensors Pix2PixModel.preprocess_input hands to the nets (CPU)."""
    import michigan_oracle as orc
    from michigan_b200.synth import synthetic_batch
    data = synthetic_batch(n or cfg["batch"], size or cfg["size"], seed if seed is not None else cfg["data_seed"])
    pre = dict(input_ref=orc.one_hot(data["label_ref"]), input_tag=orc.one_hot(data["label_tag"]),
               image_ref=data["image_ref"], image_tag=data["image_tag"], orient_mask=data["orient"], noise=data["noise"])
    return data, pre


def max_mean_abs(a, b):
    d = (a.detach().float().cpu() - b.detach().float().cpu()).abs()
    return d.max().item(), d.mean().item()
