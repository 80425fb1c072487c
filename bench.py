"""bench.py — headline benchmark of the MichiGAN hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload both|gen_fwd|train_step]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

BASELINE.json's metric has two halves, both measured by the default run and printed in ONE JSON line (rank 0):

  top level   configs[1]: generator-only forward of netG=spadeb (ngf 64), batch 8 per GPU, 512x512 synthetic inputs,
              train-mode statistics (the `generate_fake` of a training iteration: SyncBN batch statistics incl. the
              cross-rank exchange, spectral-norm power iteration), no grad.  One "step" = one forward over one batch.
  train_step  configs[2]: the full G+D train iteration (hinge GAN + GAN-feature losses, Adam TTUR), batch 8 per GPU,
              512x512 synthetic, each timed step from the same starting state; same keys as the top level (value,
              ms_per_step, e2e, roofline, gpu_launches).

  value       images/s, whole job, inputs already resident in HBM, CUDA-event timed, max over ranks: one timed block of
              exactly --steps steps between barrier + synchronize pairs, after --warmup untimed steps.
  e2e         images/s through the public API with pinned HOST buffers: H2D of the data dict and D2H of the result
              (image / loss scalars) inside the timed region
  roofline    the dominant kernel timed alone, live; roofline_worst: the kernel furthest below its roofline
  cpu_baseline / --impl reference   the reference's own CPU implementation on the host cores: the UNMODIFIED reference
              code staged under baseline/_ref (kind "reference") when present, else the CPU oracle port (kind "port")

--dump-outputs DIR writes, after the timed steps, what the last timed step returned (rank 0): DIR/gen_fwd_fake_image.npy,
DIR/train_step_generated.npy (float32) and DIR/train_step_loss_<name>.npy (float64).  Weights, inputs and Python's `random`
are seeded, so the same arguments compute from the same inputs on every run and two builds can be compared array by array.
Every step of the train leg starts from the same weights, buffers and optimizer state (see train_step_leg), so its outputs
too depend only on the arguments, up to the rounding of that one step's atomic gradient sums.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH_PER_GPU = 8
SIZE = 512
G_FWD_GFLOP_PER_IMG = 1114.2  # SURVEY.md §8d / BASELINE.md §3 (2*MAC, convs only)
TRAIN_GFLOP_PER_IMG = 4775.8  # SURVEY.md §8d: G step + D step, hinge GAN + GAN-feature losses
DUMP_MAX_BYTES = 64 * 2 ** 20
DUMP_MAX_ELEMS = 7_500_000    # per array: both 8x3x512x512 images of the default run are written whole, 60 MB together
CPU_THREADS = 32              # fixed: PyTorch's CPU convs stop scaling (and regress) beyond ~32 threads on the B200 hosts


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="both", choices=["both", "gen_fwd", "train_step", "train_step_ig"],
                    help="both (default) = generator forward + train step in one line; train_step_ig = BASELINE.json configs[4]'s "
                         "per-GPU work: the train step with --use_ig (frozen orientation-inpainting net, run twice per iteration)")
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the native path")
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ================================================================================================ CPU arm
def cpu_threads():
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, min(ncpu, CPU_THREADS))


REF_DIR = os.path.join(ROOT, "baseline", "_ref")
REF_FLAGS = ("--use_encoder --wide_edge 2 --noise_background --random_expand_mask --no_confidence_loss --no_style_loss "
             "--no_rgb_loss --no_content_loss --no_background_loss --no_vgg_loss --no_orient_loss --no_lab_loss --gpu_ids -1 "
             "--no_html --batchSize 1 --checkpoints_dir /tmp/mg_bench_ref_ckpt").split()


def reference_available():
    return os.path.isdir(os.path.join(REF_DIR, "models", "networks"))


def _reference_trainer():
    """The UNMODIFIED reference (baseline/_ref) on the CPU: its own option parser, class factory, Pix2PixTrainer."""
    from michigan_b200 import compat
    compat.stub_optional_imports()
    compat.patch_adam_betas()
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import contextlib
    import io
    import warnings
    warnings.filterwarnings("ignore", category=SyntaxWarning)
    import models.networks as networks
    compat.patch_style_content_loss(networks)
    argv = sys.argv
    sys.argv = ["bench"] + REF_FLAGS
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            from options.train_options import TrainOptions
            opt = TrainOptions().parse()
            from trainers.pix2pix_trainer import Pix2PixTrainer
            trainer = Pix2PixTrainer(opt)
    finally:
        sys.argv = argv
    return trainer


def cpu_reference_ips(steps, warmup, train=False):
    """images/s of the reference's CPU path, batch 1, 512x512, same net / synthetic inputs / deterministic weights.
    -> (gen_fwd images/s, ms per forward, train images/s or None, cores, kind)."""
    from michigan_b200.synth import fill_state_dict, synthetic_batch
    cores = cpu_threads()
    torch.set_num_threads(cores)
    data = synthetic_batch(1, SIZE, 1234)
    import random
    if reference_available():
        kind = "reference"
        trainer = _reference_trainer()
        m = trainer.pix2pix_model_on_one_gpu
        fill_state_dict(m.netG.state_dict(), 0)
        fill_state_dict(m.netD.state_dict(), 1)
        m.train()

        def fwd():
            with torch.no_grad():
                ins = m.preprocess_input(dict(data))
                m.generate_fake(ins[0], ins[2], orient_mask=ins[4], input_tag=ins[1], image_tag=ins[3], noise=ins[7])

        def train_it():
            trainer.run_generator_one_step(dict(data))
            trainer.run_discriminator_one_step(dict(data))
    else:
        kind = "port"
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import michigan_oracle as orc
        from helpers import preprocessed, reference_layout_state
        cfg = dict(ngf=64, ndf=64, size=SIZE, batch=1, data_seed=1234)
        sd = reference_layout_state("G", cfg, 0)
        _, pre = preprocessed(cfg)
        oopt = orc.default_opt(isTrain=True)

        def fwd():
            with torch.no_grad():
                orc.generate_fake(sd, oopt, pre, True, rng_k=25)
        train_it = None
    random.seed(0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        fwd()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    ips = len(times) / sum(times)
    train_ips = None
    if train and train_it is not None:
        train_it()                              # warm-up (allocations, lazy init)
        t0 = time.perf_counter()
        train_it()
        train_ips = 1.0 / (time.perf_counter() - t0)
    return ips, sum(times) / len(times) * 1e3, train_ips, cores, kind


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, min(a.steps, 5)), max(1, min(a.warmup, 1))
    want_train = a.workload in ("both", "train_step")
    ips, ms, train_ips, cores, kind = cpu_reference_ips(steps, warm, train=want_train)
    what = "the unmodified reference (baseline/_ref) imported on the CPU" if kind == "reference" else "the CPU oracle port"
    line = {
        "impl": "reference", "metric": "512x512 images/sec (generator forward)", "value": ips, "unit": "images/s",
        "n_gpus": a.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "generator-only forward (netG=spadeb ngf64, train-mode statistics, no grad), 512x512 synthetic",
                   "per_step_images": 1, "note": "CPU arm (%s): bounded sample of 1 image per step on the host cores" % what},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": "%d timed forwards of 1 image (batch 1) after %d warm-up" % (steps, warm)},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if train_ips is not None:
        line["train_step"] = {"metric": "512x512 images/sec (train step)", "value": train_ips, "unit": "images/s",
                              "ms_per_step": 1e3 / train_ips, "sample": "1 timed G+D iteration of 1 image after 1 warm-up",
                              "e2e": {"value": train_ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ================================================================================================ single-kernel rooflines
# DRAM traffic of one launch of the dominant kernel from the `ncu --set full` capture committed under profiles/
# (dram__bytes_read.sum + dram__bytes_write.sum at N=8); algorithmic bytes at N=8 (2,097,152 pixels): actv fp16 128 ch 537 MB +
# x fp32 128 ch at half resolution 268 MB + weights 0.6 MB read, bf16 hi+lo 128 ch 1074 MB written - the kernel moves its
# algorithmic bytes and nothing more.
NCU_TRAFFIC_BYTES_N8 = 809.607936e6 + 1027.305e6
NCU_TRAFFIC_SOURCE = "profiles/r02_ncu_spade_gemm_f16_tma.txt"


def _time_kernel(f, reps=5):
    flush = torch.empty(192 * 1024 * 1024 // 4, device="cuda")
    for _ in range(3):
        f()
    times = []
    for _ in range(reps):
        flush.zero_()  # evict L2 (126 MB) between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return sorted(times)[len(times) // 2]


def dominant_kernel_roofline(batch):
    """The fused SPADE gamma/beta implicit GEMM of up_3.norm_0 alone, in the operand format the forward uses
    (precision mode mixed16: fp16 operands, fp32 accumulate, bf16 hi/lo output; mode tf32: TF32 operands):
    A = actv [N,512,512,128], N_gemm = 2*128, K = 9*128, SPADE epilogue reading x [N,256,256,128] (upsample folded)
    and writing h [N,512,512,128].  FLOPs per launch = 2 * N*512*512 * 1152 * 256 (SURVEY.md Appendix A rows
    G.up_3.norm_0.mlp_gamma + mlp_beta = 2 * 77.309 GFLOP per image)."""
    from michigan_b200 import ops, precision
    dev = "cuda"
    actv = torch.randn(batch, SIZE, SIZE, 128, device=dev)
    wg = torch.randn(128, 128, 3, 3, device=dev) / 34
    xs = torch.randn(batch, SIZE // 2, SIZE // 2, 128, device=dev)
    v = torch.ones(128, device=dev)
    if precision.mode() == "tf32":
        wp = ops.pack_weight_gb(wg, wg)
        kind = "kind::tf32"
        f = lambda: ops.conv_igemm(actv, wp, 128, 3, 3, 1, 1, act=2, round_out=True, spade=(xs, 1, v, v, v, v))
    else:
        a16 = actv.half()
        wp = ops.pack_weight_gb16(wg, wg)
        kind = "kind::f16"
        f = lambda: ops.conv_igemm(a16, wp, 128, 3, 3, 1, 1, act=2, a_fmt=ops.F16, spade=(xs, 1, v, v, v, v),
                                   out16=(ops.BF16, True), want_f32=False)
    ms = _time_kernel(f)
    flops = 2.0 * batch * SIZE * SIZE * 1152 * 256
    return flops / (ms * 1e-3) / 1e12, ms, flops, kind


def worst_kernel_roofline(batch):
    """The kernel furthest below its roofline among those that matter (VERDICT r1, weak #2): the split-precision generic
    conv at its thinnest shape, up_3.conv_0 = 3x3, 128 -> 64 at 512x512 (bf16 hi+lo operands, 3 products = 2 MMAs per K
    step), 2 * N*512*512 * 1152 * 64 algorithmic FLOPs per launch (SURVEY.md Appendix A: 19.3 GF per image)."""
    from michigan_b200 import ops, precision
    dev = "cuda"
    x = torch.randn(batch, SIZE, SIZE, 128, device=dev)
    w = torch.randn(64, 128, 3, 3, device=dev) / 34
    b = torch.zeros(64, device=dev)
    if precision.mode() == "tf32":
        wp = ops.pack_weight(w, None, True)
        f = lambda: ops.conv_igemm(x, wp, 64, 3, 3, 1, 1, bias=b)
        kind = "kind::tf32, one pass"
    else:
        hi = x.bfloat16()
        lo = (x - hi.float()).bfloat16()
        wp = ops.pack_weight16(w, None, ops.BF16, split=True)
        f = lambda: ops.conv_igemm(hi, wp, 64, 3, 3, 1, 1, bias=b, a_fmt=ops.BF16, x_lo=lo)
        kind = "kind::f16 bf16 hi+lo split"
    ms = _time_kernel(f)
    flops = 2.0 * batch * SIZE * SIZE * 1152 * 64
    return flops / (ms * 1e-3) / 1e12, ms, flops, kind


def wgrad_kernel_roofline(batch):
    """Dominant kernel of the train step: the weight-gradient GEMM, at the shape of the SPADE gamma|beta wgrad of up_3
    (dY = dgamma|dbeta [N,512,512,256], X = actv [N,512,512,128], 3x3): 2 * N*512*512 * 1152 * 256 FLOPs per launch, in the operand
    format the train step uses for it (precision.grad_fmt(): bf16 in mixed16 mode, TF32 otherwise)."""
    from michigan_b200 import ops, precision
    dev = "cuda"
    dy = torch.randn(batch, SIZE, SIZE, 256, device=dev)
    x = torch.randn(batch, SIZE, SIZE, 128, device=dev)
    if precision.grad_fmt() == ops.BF16:
        dy16, x16 = dy.bfloat16(), x.bfloat16()
        del dy, x
        f = lambda: ops.conv_wgrad16(dy16, x16, 3, 3, 1, 1)
        kind = "kind::f16 (bf16 operands)"
    else:
        f = lambda: ops.conv_wgrad(dy, x, 3, 3, 1, 1)
        kind = "kind::tf32"
    ms = _time_kernel(f, reps=3)
    flops = 2.0 * batch * SIZE * SIZE * 1152 * 256
    return flops / (ms * 1e-3) / 1e12, ms, flops, kind


# ================================================================================================ native arm
def timed_block(step, steps, world):
    """[barrier+sync | e0 | `steps` x step | e1 | barrier+sync] -> (device time of the block in ms, max over ranks; host time
    in ms to ISSUE the block, which has no synchronisation inside)."""
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    host_ms = (time.perf_counter() - t0) * 1e3
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), host_ms


def host_array(t, dtype):
    """`t` as a host numpy array of `dtype`; above DUMP_MAX_ELEMS elements, a sample of its flattened values at fixed seeded
    positions (the same on every run)."""
    f = t.detach().to(dtype)
    if f.numel() > DUMP_MAX_ELEMS:
        idx = torch.randperm(f.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
        f = f.reshape(-1)[idx.to(f.device)]
    return f.cpu().numpy()


def write_dump(path, arrays):
    import numpy as np
    total = sum(v.nbytes for v in arrays.values())
    assert total <= DUMP_MAX_BYTES, "dump of %d bytes exceeds %d" % (total, DUMP_MAX_BYTES)
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + ".npy"), v)


INPUT_KEYS = ("label_ref", "label_tag", "image_ref", "image_tag", "orient", "noise")


def gen_fwd_leg(a, rank, world, local, model, dump):
    """-> dict of the top-level keys of the JSON line; with --dump-outputs, rank 0 adds the last timed step's image to `dump`."""
    import torch.distributed as dist
    from michigan_b200 import _lib, precision
    from michigan_b200.synth import synthetic_batch
    batch = a.batch
    data = synthetic_batch(batch, SIZE, 1234 + rank)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in data.items()}
    host_out = torch.empty(batch, 3, SIZE, SIZE).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        pre = model.preprocess_input(host)
        torch.cuda.synchronize()
        last = {}

        def step():
            last["fake"] = model.generate_fake(pre[0], pre[2], pre[4], pre[1], pre[3], pre[5])

        for _ in range(a.warmup):
            step()
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        l0 = _lib.launch_count()
        ms_block, _ = timed_block(step, a.steps, world)
        launches = _lib.launch_count() - l0
        clocks = sampler.stop() if rank == 0 else None
        if a.dump_outputs and rank == 0:
            dump["gen_fwd_fake_image"] = host_array(last["fake"], torch.float32)

        # ---- end to end through the public API with host buffers.  Every step copies its inputs from pinned host memory
        # and reads its result back into pinned host memory; like a prefetching data loader the copies run on a second
        # stream (double-buffered), so step i+1's H2D and step i-1's D2H overlap step i's kernels.
        copy_stream = torch.cuda.Stream()
        main_stream = torch.cuda.current_stream()
        host_outs = [host_out, torch.empty_like(host_out).pin_memory()]
        tensor_keys = [k for k, v in host.items() if torch.is_tensor(v)]
        dev_sets = [{k: torch.empty_like(host[k], device="cuda") for k in tensor_keys} for _ in range(2)]

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                for k in tensor_keys:
                    dev_sets[i & 1][k].copy_(host[k], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            dev = dict(host)
            dev.update(dev_sets[i & 1])
            return dev, ev

        def e2e_run(nsteps):
            nxt = prefetch(0)
            for i in range(nsteps):
                dev, ev = nxt
                main_stream.wait_event(ev)
                if i + 1 < nsteps:
                    nxt = prefetch(i + 1)   # queued behind step i-1's read-back, which waited for step i-1's kernels
                img = model(dev, mode="inference")
                done = torch.cuda.Event()
                done.record(main_stream)
                img.record_stream(copy_stream)
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(done)
                    host_outs[i & 1].copy_(img, non_blocking=True)
            copy_stream.synchronize()
            main_stream.synchronize()

        e2e_run(max(2, a.warmup // 2 + 1))
        e2e_steps = a.steps
        barrier()
        t0 = time.perf_counter()
        e2e_run(e2e_steps)
        barrier()
        t_e2e = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        t_e2e = t_e2e.item()

    h2d = sum(v.numel() * v.element_size() for k, v in host.items() if torch.is_tensor(v) and k in INPUT_KEYS)
    d2h = host_out.numel() * 4
    ms_step = ms_block / a.steps
    return {
        "metric": "512x512 images/sec (generator forward)", "value": world * batch * a.steps / (ms_block * 1e-3), "unit": "images/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE_NOTE[precision.mode()], "data": "synthetic",
        "config": {"workload": "generator-only forward (netG=spadeb ngf64, 109.5M params, train-mode statistics, no grad), "
                               "batch %d/GPU, 512x512 synthetic mask/orient/ref inputs" % batch,
                   "global_batch": batch * world, "parallelism": "dp%d" % world,
                   "l2": "no explicit flush: each step streams multi-GB NHWC activations (>> 126 MB L2)",
                   "algorithmic_gflop_per_image": G_FWD_GFLOP_PER_IMG,
                   "timing": "one block of %d steps after %d warm-up steps" % (a.steps, a.warmup)},
        "achieved_tflops_step": G_FWD_GFLOP_PER_IMG * batch / ms_step,
        "e2e": {"value": world * batch * e2e_steps / t_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps,
                "how": "Pix2PixModel(data, mode='inference') per step; pinned host inputs -> device and image -> pinned host every "
                       "step, copies double-buffered on a second stream (prefetching-loader style), wall clock"},
        "gpu_launches": launches, "clocks": clocks,
    }


def train_step_leg(a, rank, world, local, model, dump, use_ig=False):
    """BASELINE.json configs[2]: one generator update + one discriminator update per step (train.py:94-101).  With
    --dump-outputs, rank 0 adds the last timed step's generated image and losses to `dump`."""
    import torch.distributed as dist
    from michigan_b200 import _lib
    from michigan_b200.networks.sync_batchnorm import DataParallelWithCallback, exchange_backend
    from michigan_b200.pix2pix_model import train_iteration
    from michigan_b200.synth import synthetic_batch
    batch = a.batch
    wrap = DataParallelWithCallback(model, device_ids=[local])
    optG, optD = model.create_optimizers(model.opt)
    data = synthetic_batch(batch, SIZE, 1234 + rank, use_ig=use_ig)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in data.items()}
    dev = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in data.items()}
    last = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Every step of the timed leg starts from the same state: weights and buffers of G and D, zeroed Adam moments and step
    # counts, and Python's `random`.  The gradient sums accumulate with float atomics, and Adam turns their last-bit
    # differences into different updates, so a state carried from step to step would make what the n-th step computes drift
    # from run to run.  Restoring is one device copy of the model state per step (~0.5 GB), small beside the step itself.
    for opt in (optG, optD):        # create the Adam state now: a zero gradient leaves the weights and moments unchanged
        for group in opt.param_groups:
            for p in group["params"]:
                p.grad = torch.zeros_like(p)
        opt.step()
        opt.zero_grad(set_to_none=True)

    def by_kind(tensors):           # one fused foreach launch per (device, dtype)
        kinds = {}
        for t in tensors:
            kinds.setdefault((t.device, t.dtype), []).append(t)
        return list(kinds.values())

    model_state = by_kind(t for net in (model.netG, model.netD) for t in net.state_dict().values())
    saved_state = [[t.clone() for t in ts] for ts in model_state]
    adam_state = by_kind(v for opt in (optG, optD) for s in opt.state.values() for v in s.values() if torch.is_tensor(v))
    saved_random = random.getstate()

    def restore():
        for dst, src in zip(model_state, saved_state):
            torch._foreach_copy_(dst, src)
        for ts in adam_state:
            torch._foreach_zero_(ts)
        random.setstate(saved_random)

    def step():
        restore()
        g, d, generated = train_iteration(wrap, optG, optD, dict(dev))
        last["losses"], last["generated"] = {**g, **d}, generated

    for _ in range(a.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ms_block, host_block_ms = timed_block(step, a.steps, world)
    host_ms = host_block_ms / a.steps
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump["train_step_generated"] = host_array(last["generated"], torch.float32)
        for k, v in last["losses"].items():
            dump["train_step_loss_" + k] = host_array(v, torch.float64)

    # ---- end to end: every step's inputs come from pinned HOST tensors (copied on a second stream into one of two device
    # buffers while the previous step computes - a prefetching loader) and every step ends with its loss scalars read back to the
    # host and a stream synchronisation
    loss_host = torch.empty(8, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream()
    main_stream = torch.cuda.current_stream()
    tensor_keys = [k for k, v in host.items() if torch.is_tensor(v)]
    dev_sets = [{k: torch.empty_like(host[k], device="cuda") for k in tensor_keys} for _ in range(2)]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            for k in tensor_keys:
                dev_sets[i & 1][k].copy_(host[k], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        d = dict(host)
        d.update(dev_sets[i & 1])
        return d, ev

    def e2e_run(nsteps):
        nxt = prefetch(0)
        nl = 0
        for i in range(nsteps):
            d, ev = nxt
            main_stream.wait_event(ev)
            if i + 1 < nsteps:
                nxt = prefetch(i + 1)        # buffer (i+1)&1 was last read by step i-1, which has been synchronised
            g, dl, _ = train_iteration(wrap, optG, optD, d)
            vals = torch.stack([v.detach().mean() for v in {**g, **dl}.values()])
            nl = vals.numel()
            loss_host[:nl].copy_(vals, non_blocking=True)
            main_stream.synchronize()
        return nl

    e2e_run(2)
    e2e_steps = a.steps
    barrier()
    t0 = time.perf_counter()
    nl = e2e_run(e2e_steps)
    barrier()
    t_e2e = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    t_e2e = t_e2e.item()
    keys = INPUT_KEYS + (("hole", "orient_rgb") if use_ig else ())
    h2d = sum(v.numel() * v.element_size() for k, v in host.items() if torch.is_tensor(v) and k in keys)
    ms_step = ms_block / a.steps
    out = {
        "metric": "512x512 images/sec (train step%s)" % (", --use_ig" if use_ig else ""), "value": world * batch * a.steps / (ms_block * 1e-3),
        "unit": "images/s", "vs_baseline": None, "data": "synthetic",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "dtype": "forward: fp16/bf16 tensor-core operands as the generator-forward leg; gradient GEMMs of the generator blocks: bf16 operands "
                 "(encoders / discriminator: TF32); fp32 accumulate, storage, statistics and Adam",
        "config": {"workload": "full G+D train iteration (hinge GAN + GAN-feature losses, Adam TTUR), netG=spadeb ngf64, "
                               "netD=multiscale ndf64, batch %d/GPU, 512x512 synthetic" % batch,
                   "global_batch": batch * world, "parallelism": "dp%d" % world,
                   "l2": "no explicit flush: multi-GB activations per step",
                   "algorithmic_gflop_per_image": TRAIN_GFLOP_PER_IMG + (2 * 151.9 if use_ig else 0.0),
                   "use_ig": bool(use_ig),
                   "timing": "one block of %d steps after %d warm-up steps" % (a.steps, a.warmup),
                   "syncbn_exchange": exchange_backend(), "grad_allreduce": "in-backward staged NCCL all-reduce (AVG) of a flat fp32 buffer"},
        "achieved_tflops_step": (TRAIN_GFLOP_PER_IMG + (2 * 151.9 if use_ig else 0.0)) * batch / ms_step,
        "e2e": {"value": world * batch * e2e_steps / t_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * nl,
                "steps": e2e_steps,
                "how": "train_iteration(DataParallelWithCallback(Pix2PixModel), ...) per step; inputs pinned host -> device every step on a "
                       "second stream (double-buffered), loss scalars -> pinned host and a stream synchronisation every step; wall clock"},
        "gpu_launches": launches, "clocks": clocks, "host_enqueue_ms_per_step": host_ms,
        "losses": {k: float(v.detach().mean()) for k, v in last["losses"].items()},
    }
    return out


def run_native(a):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from michigan_b200.options import make_opt
    from michigan_b200.pix2pix_model import Pix2PixModel
    from michigan_b200.synth import fill_state_dict

    torch.manual_seed(0)
    random.seed(0)   # the training-mode generator draws its mask dilation with Python's `random`, as the reference does
    use_ig = a.workload == "train_step_ig"
    extra = {}
    if use_ig:
        # a random-init InpaintingModel_gen.pth in the reference's layout ({'generator': state_dict}, util.py:245-257)
        import tempfile
        from michigan_b200.networks import InpaintGenerator
        ckdir = os.path.join(tempfile.gettempdir(), "mg_bench_ig_%d" % os.getpid())
        os.makedirs(os.path.join(ckdir, "MichiGAN"), exist_ok=True)
        ig = InpaintGenerator()
        fill_state_dict(ig.state_dict(), 2)
        torch.save({"generator": ig.state_dict()}, os.path.join(ckdir, "MichiGAN", "InpaintingModel_gen.pth"))
        extra = dict(use_ig=True, checkpoints_dir=ckdir, name="MichiGAN", ig_model_name="InpaintingModel_gen.pth", netIG="inpaint")
    opt = make_opt(is_train=True, gpu_ids=[local], batchSize=a.batch * world, niter=50, niter_decay=0, **extra)
    model = Pix2PixModel(opt)
    fill_state_dict(model.netG.state_dict(), 0)  # random-init weights of the reference architecture (109.5 M params)
    fill_state_dict(model.netD.state_dict(), 1)
    model.train()

    line = None
    dump = {}
    if a.workload in ("both", "gen_fwd"):
        line = gen_fwd_leg(a, rank, world, local, model, dump)
    train = None
    if a.workload in ("both", "train_step", "train_step_ig"):
        train = train_step_leg(a, rank, world, local, model, dump, use_ig)
    if rank == 0:
        if a.dump_outputs:
            write_dump(a.dump_outputs, dump)
        pk, pk_kind = peaks()
        peak_tf = float(pk["bf16_tflops"])
        if line is not None:
            tf, kms, kflops, kkind = dominant_kernel_roofline(a.batch)
            line["roofline"] = {
                "kernel": "igemm_tf32_kernel<1,16> (fused SPADE gamma|beta implicit GEMM + modulate + LeakyReLU, up_3.norm_0 shape, tcgen05 %s)" % kkind,
                "bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                "traffic": NCU_TRAFFIC_BYTES_N8 * a.batch / 8 if kkind == "kind::f16" else None,
                "traffic_unit": "bytes per launch (dram read + write, ncu --set full, %s)" % NCU_TRAFFIC_SOURCE,
                "peak_kind": "%s bf16 dense burst (MEASURED_PEAKS.json)%s" % (
                    pk_kind, "; kind::tf32 issues at half the bf16 rate" if kkind == "kind::tf32" else ""),
                "ms_per_launch": kms, "flops_per_launch": kflops}
            wtf, wms, wflops, wkind = worst_kernel_roofline(a.batch)
            line["roofline_worst"] = {
                "kernel": "conv3x3_group_kernel<0,16> (3x3 implicit-GEMM conv on the halo-patch + M-tile-group schedule, up_3.conv_0 shape 128->64 at 512x512, %s)" % wkind,
                "bound": "tensor", "achieved": wtf, "peak": peak_tf, "unit": "TFLOP/s", "frac": wtf / peak_tf, "traffic": None,
                "note": "algorithmic FLOPs (one product per MAC); the split-precision form issues 3 products per MAC",
                "ms_per_launch": wms, "flops_per_launch": wflops}
        if train is not None:
            gtf, gms, gflops, gkind = wgrad_kernel_roofline(a.batch)
            train["roofline"] = {
                "kernel": "wgrad_tf32_kernel (weight-gradient GEMM, SPADE gamma|beta wgrad of up_3: K = N*512*512 pixels, 256 x 1152 outputs, "
                          "MN-major operands, tcgen05 %s)" % gkind,
                "bound": "tensor", "achieved": gtf, "peak": peak_tf, "unit": "TFLOP/s", "frac": gtf / peak_tf, "traffic": None,
                "peak_kind": "%s bf16 dense burst (MEASURED_PEAKS.json)" % pk_kind,
                "ms_per_launch": gms, "flops_per_launch": gflops}
        if line is None:
            line = train
        elif train is not None:
            train.pop("clocks_unused", None)
            line["train_step"] = train
        if not a.no_cpu_baseline and world == 1:
            ips, ms_cpu, train_ips, cores, kind = cpu_reference_ips(3, 1, train=False)
            line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
                                    "sample": "3 timed generator forwards of 1 image (batch 1, same net/size) after 1 warm-up"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DTYPE_NOTE = {
    "mixed16": "fp16/bf16 tensor-core operands (bf16 hi+lo split where needed), fp32 accumulate and storage",
    "tf32": "tf32",
}


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_native(args)
