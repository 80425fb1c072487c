"""Generate the golden fixtures from the LIVE reference (run in the build container only):

    python tests/golden/make_golden.py

For each case the unmodified reference modules (/root/reference, imported through ref_shims.py) and
the CPU oracle (oracle/michigan_oracle.py) are run on identical deterministic weights
(michigan_b200.synth.fill_state_dict) and inputs (synthetic_batch); the script ASSERTS that they agree
(fp32 reassociation noise only) and stores the reference's outputs in tests/golden/*.npz.  The
fixtures are what pins the oracle (tests/test_oracle_golden.py) and the CUDA path
(tests/test_gpu_parity.py) wherever the reference itself is not available.
"""
import json
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import ref_shims  # noqa: E402
import michigan_oracle as orc  # noqa: E402
from michigan_b200.synth import fill_state_dict, synthetic_batch  # noqa: E402

CFG = dict(ngf=64, ndf=64, size=128, batch=2, seed_G=11, seed_D=12, data_seed=77, py_seed=5)
TOL = 2e-5


def summary(t, stride=37, cap=4096):
    """Full statistics + a strided subsample: small, but any localized error moves them."""
    f = t.detach().float().reshape(-1)
    return np.concatenate([np.array([f.mean().item(), f.std().item(), f.abs().max().item(), f.abs().mean().item()],
                                    dtype=np.float64).astype(np.float32), f[::stride][:cap].numpy()])


def check(name, ref, got, tol=TOL):
    err = (ref - got).abs().max().item()
    scale = max(ref.abs().max().item(), 1e-6)
    print("  %-34s max|ref-oracle| %.2e (ref max %.2e)" % (name, err, scale))
    assert err <= tol * max(scale, 1.0), "oracle disagrees with the reference on %s: %g" % (name, err)


def rng_k(size, py_seed):
    random.seed(py_seed)
    th = int(size * 0.05)
    th = th if th % 2 == 1 else th + 1
    return random.choice([max(th - 4, 1), max(th - 2, 1), th, th + 2, th + 4])


def main():
    torch.set_num_threads(8)
    torch.manual_seed(0)
    ref_shims.patch_training()
    c = CFG
    size = c["size"]
    extra = ["--ngf", str(c["ngf"]), "--ndf", str(c["ndf"]), "--crop_size", str(size), "--load_size", str(size),
             "--batchSize", str(c["batch"])]
    opt = ref_shims.ref_options(True, extra)
    from trainers.pix2pix_trainer import Pix2PixTrainer
    trainer = Pix2PixTrainer(opt)
    model = trainer.pix2pix_model
    netG, netD = model.netG, model.netD
    fill_state_dict(netG.state_dict(), c["seed_G"])
    fill_state_dict(netD.state_dict(), c["seed_D"])
    sdG0 = {k: v.clone() for k, v in netG.state_dict().items()}
    sdD0 = {k: v.clone() for k, v in netD.state_dict().items()}
    oopt = orc.default_opt(ngf=c["ngf"], ndf=c["ndf"], crop_size=size, isTrain=True)
    out = {"config": np.frombuffer(json.dumps(c).encode(), dtype=np.uint8)}

    data = synthetic_batch(c["batch"], size, c["data_seed"])
    input_ref, input_tag, image_ref, image_tag, orient_mask, hole, orient_rgb, noise = model.preprocess_input(dict(data))
    pre = dict(input_ref=input_ref, input_tag=input_tag, image_ref=image_ref, image_tag=image_tag, orient_mask=orient_mask,
               noise=noise)

    # ------------------------------------------------------------------ G forward, train mode (batch stats)
    print("[G train-mode forward]")
    taps_ref = {}
    hooks = []
    for name in ["fc", "head_0", "G_middle_0", "G_middle_1", "up_0", "up_1", "up_2", "up_3"]:
        key = name + "_pre" if name.startswith("up_") else name
        def tap_hook(m, i, o, key=key):
            taps_ref[key] = o.detach().clone()

        hooks.append(getattr(netG, name).register_forward_hook(tap_hook))
    def bg_hook(m, i, o):
        for j, f in enumerate(o[0]):
            taps_ref["bg%d" % j] = f.detach().clone()

    hooks.append(netG.backgroud_enc.register_forward_hook(bg_hook))
    k = rng_k(size, c["py_seed"])
    random.seed(c["py_seed"])
    netG.train()
    with torch.no_grad():
        g_train, _, _ = model.generate_fake(input_ref, image_ref, orient_mask=orient_mask, input_tag=input_tag,
                                            image_tag=image_tag, noise=noise)
    for h in hooks:
        h.remove()
    sdG_o = {kk: v.clone() for kk, v in sdG0.items()}
    taps_o = {}
    with torch.no_grad():
        g_train_o = orc.generate_fake(sdG_o, oopt, pre, True, rng_k=k, taps=taps_o)
    check("G output (train mode)", g_train, g_train_o)
    for name, t in taps_ref.items():
        check("tap " + name, t, taps_o[name])
    sdG1 = {kk: v.clone() for kk, v in netG.state_dict().items()}
    for kk in sdG1:
        if kk.endswith(("running_mean", "running_var", "weight_u", "weight_v")):
            check("post-forward " + kk[-40:], sdG1[kk], sdG_o[kk], 1e-5) if kk.endswith("weight_u") and "up_3" in kk else None
            assert torch.allclose(sdG1[kk], sdG_o[kk], atol=2e-5, rtol=1e-4), kk
        if kk.endswith("num_batches_tracked"):
            assert int(sdG1[kk]) == 0
    out["rng_k"] = np.array([k])
    out["g_train_out"] = g_train.numpy()
    for name in taps_o:
        out["tap/" + name] = summary(taps_o[name] if name not in taps_ref else taps_ref[name])
    for kk, v in sdG1.items():
        if kk.endswith(("running_mean", "running_var", "weight_u", "weight_v")):
            out["g_post/" + kk] = v.numpy()

    # ------------------------------------------------------------------ G forward, eval mode (inference.py flow)
    print("[G eval-mode forward (TestOptions / mode='inference')]")
    topt = ref_shims.ref_options(False, ["--ngf", str(c["ngf"]), "--crop_size", str(size), "--load_size", str(size)])
    from models.pix2pix_model import Pix2PixModel
    tmodel = Pix2PixModel(topt)
    tmodel.eval()
    tmodel.netG.load_state_dict(sdG1)
    g_eval = tmodel(dict(data), mode="inference")
    oopt_e = orc.default_opt(ngf=c["ngf"], crop_size=size, isTrain=False)
    sdG_e = {kk: v.clone() for kk, v in sdG1.items()}
    with torch.no_grad():
        g_eval_o = orc.generate_fake(sdG_e, oopt_e, pre, False)
    check("G output (eval mode)", g_eval, g_eval_o)
    for kk in sdG_e:
        assert torch.equal(sdG_e[kk], sdG1[kk]), "eval forward must not touch state: " + kk
    out["g_eval_out"] = g_eval.numpy()

    # ------------------------------------------------------------------ D forward (train mode)
    print("[D forward]")
    fake_and_real = torch.cat([torch.cat([input_tag, orc.orient_channels(orient_mask, input_tag[:, 1:2], oopt), g_train], 1),
                               torch.cat([input_tag, orc.orient_channels(orient_mask, input_tag[:, 1:2], oopt), image_tag], 1)], 0)
    netD.train()
    with torch.no_grad():
        d_ref = netD(fake_and_real)
    sdD_o = {kk: v.clone() for kk, v in sdD0.items()}
    with torch.no_grad():
        d_o = orc.multiscale_discriminator(fake_and_real, sdD_o, oopt, True)
    for i in range(2):
        for j in range(5):
            check("D[%d][%d] %s" % (i, j, tuple(d_ref[i][j].shape)), d_ref[i][j], d_o[i][j])
            out["d/%d/%d" % (i, j)] = d_ref[i][j].numpy() if j == 4 else summary(d_ref[i][j])
    sdD1 = {kk: v.clone() for kk, v in netD.state_dict().items()}
    for kk, v in sdD1.items():
        if kk.endswith(("weight_u", "weight_v")):
            assert torch.allclose(v, sdD_o[kk], atol=2e-5, rtol=1e-4), kk
            out["d_post/" + kk] = v.numpy()

    # ------------------------------------------------------------------ one G step + one D step (trainer)
    print("[train iteration: G step, D step]")
    netG.load_state_dict(sdG0)
    netD.load_state_dict(sdD0)
    random.seed(c["py_seed"])
    trainer.run_generator_one_step(dict(data))
    g_losses = {kk: float(v.mean()) for kk, v in trainer.g_losses.items()}
    gradsG = {n: p.grad.detach().clone() for n, p in netG.named_parameters() if p.grad is not None}
    # oracle: same step through autograd on the functional restatement
    sdG_s = {kk: v.clone() for kk, v in sdG0.items()}
    sdD_s = {kk: v.clone() for kk, v in sdD0.items()}
    pnames = [n for n, _ in netG.named_parameters()]
    for n in pnames:
        sdG_s[n].requires_grad_(True)
    losses_o, fake_o = orc.compute_generator_loss(sdG_s, sdD_s, oopt, pre, rng_k=k)
    orc.trainer_loss(losses_o).backward()
    for kk in g_losses:
        print("  G loss %-10s ref %.6f oracle %.6f" % (kk, g_losses[kk], float(losses_o[kk].mean())))
        assert abs(g_losses[kk] - float(losses_o[kk].mean())) <= 1e-5 * max(1.0, abs(g_losses[kk]))
    worst = 0.0
    for n in pnames:
        if n not in gradsG:   # backgroud_enc.layer4 is never executed (encoder.py:284 vs 323-330)
            assert sdG_s[n].grad is None, n
            continue
        g_ref, g_o = gradsG[n], sdG_s[n].grad
        # biases that feed a BatchNorm have mathematically zero gradient (1e-9 noise): absolute floor
        rel = (g_ref - g_o).abs().max().item() / max(g_ref.abs().max().item(), 1e-5)
        if rel > 5e-3:
            print("    grad mismatch %-45s ref max %.3e  err %.3e" % (n, g_ref.abs().max().item(), (g_ref - g_o).abs().max().item()))
        worst = max(worst, rel)
    print("  G grads: worst relative max-error over %d tensors: %.2e" % (len(pnames), worst))
    assert worst < 5e-3, worst
    out["g_losses"] = np.array([g_losses["GAN"], g_losses["GAN_Feat"]], dtype=np.float64)
    for n in ["conv_img.weight", "up_3.conv_1.weight_orig", "up_3.norm_1.mlp_gamma.weight", "up_0.norm_s.mlp_shared.0.weight",
              "head_0.conv_0.weight_orig", "fc.layer1.weight", "backgroud_enc.layer2.conv.weight", "up_1.conv_s.weight_orig",
              "G_middle_1.norm_0.mlp_beta.bias", "up_2.conv_0.bias"]:
        out["g_grad/" + n] = summary(gradsG[n], stride=101)
    sdG2 = {kk: v.clone() for kk, v in netG.state_dict().items()}
    for n in ["conv_img.weight", "up_3.conv_1.weight_orig", "head_0.norm_0.mlp_gamma.weight"]:
        out["g_post_step/" + n] = summary(sdG2[n], stride=101)

    random.seed(c["py_seed"] + 1)
    k2 = rng_k(size, c["py_seed"] + 1)
    random.seed(c["py_seed"] + 1)
    trainer.run_discriminator_one_step(dict(data))
    d_losses = {kk: float(v.mean()) for kk, v in trainer.d_losses.items()}
    gradsD = {n: p.grad.detach().clone() for n, p in netD.named_parameters() if p.grad is not None}
    sdG_s2 = {kk: v.clone() for kk, v in sdG2.items()}       # G after its optimizer step and its train-mode forward
    sdD_s2 = {kk: v.clone() for kk, v in sdD_s.items()}      # D u/v after the G step's D forward; weights unchanged
    for kk in sdD_s2:
        sdD_s2[kk] = sdD_s2[kk].detach().clone()
    dnames = [n for n, _ in netD.named_parameters()]
    for n in dnames:
        sdD_s2[n].requires_grad_(True)
    dl_o = orc.compute_discriminator_loss(sdG_s2, sdD_s2, oopt, pre, rng_k=k2)
    orc.trainer_loss(dl_o).backward()
    for kk in d_losses:
        print("  D loss %-10s ref %.6f oracle %.6f" % (kk, d_losses[kk], float(dl_o[kk].mean())))
        assert abs(d_losses[kk] - float(dl_o[kk].mean())) <= 2e-5 * max(1.0, abs(d_losses[kk]))
    worst = 0.0
    for n in dnames:
        # relative L2: the hinge loss is piecewise linear, a logit within 1e-6 of the kink flips its
        # gradient mask between two fp32 evaluation orders, which moves single elements, not the norm
        rel = (gradsD[n] - sdD_s2[n].grad).norm().item() / max(gradsD[n].norm().item(), 1e-5)
        if rel > 5e-3:
            print("    D grad mismatch %-40s ref max %.3e err %.3e" % (n, gradsD[n].abs().max().item(), (gradsD[n] - sdD_s2[n].grad).abs().max().item()))
        worst = max(worst, rel)
    print("  D grads: worst relative L2 error over %d tensors: %.2e" % (len(dnames), worst))
    assert worst < 2e-2, worst
    out["rng_k2"] = np.array([k2])
    out["d_losses"] = np.array([d_losses["D_Fake"], d_losses["D_real"]], dtype=np.float64)
    for n in dnames:
        out["d_grad/" + n] = summary(gradsD[n], stride=53)

    # ------------------------------------------------------------------ D step from the INITIAL weights
    # (decoupled from the generator's Adam update, whose first step is sign-like and amplifies noise)
    print("[D step from initial weights]")
    netG.load_state_dict(sdG0)
    netD.load_state_dict(sdD0)
    random.seed(c["py_seed"] + 2)
    k3 = rng_k(size, c["py_seed"] + 2)
    random.seed(c["py_seed"] + 2)
    trainer.run_discriminator_one_step(dict(data))
    d0_losses = {kk: float(v.mean()) for kk, v in trainer.d_losses.items()}
    gradsD0 = {n: p.grad.detach().clone() for n, p in netD.named_parameters() if p.grad is not None}
    sdG_s3 = {kk: v.clone() for kk, v in sdG0.items()}
    sdD_s3 = {kk: v.clone() for kk, v in sdD0.items()}
    for n in dnames:
        sdD_s3[n].requires_grad_(True)
    dl3 = orc.compute_discriminator_loss(sdG_s3, sdD_s3, oopt, pre, rng_k=k3)
    orc.trainer_loss(dl3).backward()
    for kk in d0_losses:
        print("  D loss %-10s ref %.6f oracle %.6f" % (kk, d0_losses[kk], float(dl3[kk].mean())))
        assert abs(d0_losses[kk] - float(dl3[kk].mean())) <= 2e-5 * max(1.0, abs(d0_losses[kk]))
    worst = max((gradsD0[n] - sdD_s3[n].grad).norm().item() / max(gradsD0[n].norm().item(), 1e-5) for n in dnames)
    print("  D grads (initial weights): worst relative L2 error %.2e" % worst)
    assert worst < 2e-2, worst
    out["rng_k3"] = np.array([k3])
    out["d0_losses"] = np.array([d0_losses["D_Fake"], d0_losses["D_real"]], dtype=np.float64)
    for n in dnames:
        out["d0_grad/" + n] = summary(gradsD0[n], stride=53)

    # two files, each under 1 MB: the network outputs and losses, and the intermediate / post-step state and gradients
    state = ("tap/", "g_post", "d_post", "g_grad/", "d_grad/", "d0_grad/")
    for name, part in (("golden_ngf64_128.npz", {k: v for k, v in out.items() if not k.startswith(state)}),
                       ("golden_ngf64_128_state.npz", {k: v for k, v in out.items() if k.startswith(state)})):
        path = os.path.join(HERE, name)
        np.savez_compressed(path, **part)
        print("wrote %s (%.1f KB, %d arrays)" % (path, os.path.getsize(path) / 1024, len(part)))


if __name__ == "__main__":
    main()
