#!/usr/bin/env python
"""bench.py — restored 256x256 images/sec @100 DDIM steps (BASELINE.json metric), one JSON line.

Default workload (BASELINE configs[1], `--config 2`): celeba_hq.yml denoiser (random init, seed 1234) x SuperResolution(4x average
pooling), sigma_y=0, T_sampling=100, eta=0.85, 16 images per GPU.  A "step" = one full sampling of the per-GPU batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5a|5b] [--precision fp32|fp16]
                    [--dump-outputs DIR]

`value`  : the loop with x_T / y resident in HBM; the per-pair Gaussian draws ARE inside the timed region (drawn chunk by chunk on a
           side stream by ddnm_b200.sampler, like the reference's one randn_like per step).
`e2e`    : the public drop-in call (ddnm_diffusion / ddnm_plus_diffusion) with pinned HOST x_T / y and CPU results.
N>1 is launched by torchrun (one rank per GPU): rows shard over ranks, no traffic inside the loop, one all-gather of the restored
images per step (weak scaling); an untimed sharded-vs-unsharded check runs first (`shard_check`).
`--dump-outputs DIR`: after the timed steps, the last step's results (restored images `x0`, last x0 prediction `x0_pred`, all
ranks' rows) go to DIR/<name>.npy as float32, so that two builds can be compared output for output: every input is drawn from fixed
seeds, so the same arguments give the same inputs.  An output over its share of 64 MB is replaced by a fixed, seeded sample of its
elements (flattened).
`--impl reference` times the UNMODIFIED reference (oracle/_ref, see oracle/make_ref.py) on the host cores on a bounded sample.
The other BASELINE configs (`--config 3|4|5a|5b`) and the fp16 fast mode print the same line for their workload; their results are
kept under profiles/ (the driver's N=1 line stays configs[1]).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "images/sec"
ETA, RES = 0.85, 256
CONFIGS = {
    # key: BASELINE.json configs index + 1 (SURVEY section 8d numbering)
    "2": dict(net="celeba", op="sr4", T=100, tl=1, tr=1, sigma_y=0.0, B=16,
              workload="celeba_hq.yml simple-UNet (113.7M params, random init seed 1234) + sr_averagepooling x4, sigma_y=0, T_sampling=100, eta=0.85, batch 16/GPU"),
    "3": dict(net="imagenet", op="color", T=100, tl=1, tr=1, sigma_y=0.0, B=8,
              workload="imagenet_256.yml UNetModel (552.8M params, random init seed 1234, learn_sigma) + colorization, sigma_y=0, T_sampling=100, eta=0.85, batch 8/GPU (64 over 8 GPUs)"),
    "4": dict(net="imagenet", op="inpaint", T=100, tl=3, tr=3, sigma_y=0.1, B=8,
              workload="imagenet_256.yml UNetModel + inpainting (exp/inp_masks/mask.npy), DDNM+ sigma_y=0.05 (0.1 internal), T_sampling=100, travel_length=3, travel_repeat=3 (298 UNet evals + 198 travel-back pairs), batch 8/GPU"),
    "5a": dict(net="celeba", op="deblur", T=250, tl=1, tr=1, sigma_y=0.0, B=16,
               workload="celeba_hq.yml simple-UNet + deblur_gauss (sigma 10, 5 taps), sigma_y=0, T_sampling=250, batch 16/GPU (128 over 8 GPUs)"),
    "5b": dict(net="celeba", op="wh", T=250, tl=1, tr=1, sigma_y=0.0, B=16,
               workload="celeba_hq.yml simple-UNet + cs_walshhadamard ratio 0.25, sigma_y=0, T_sampling=250, batch 16/GPU (128 over 8 GPUs)"),
}
STEP_KERNELS = {"sr4": 1, "color": 1, "inpaint": 1, "wh": 7, "deblur": 13}   # own launches of the fused per-pair update (operators.cu step())
DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Write each tensor of `arrays` as dirname/<name>.npy (float32), in all at most DUMP_BYTES: a tensor larger than its share is
    replaced by the elements at a fixed, seeded set of flat positions (in ascending order), the same in every run."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096          # room for the .npy header
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            idx = np.random.default_rng(1234).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(dirname, name + ".npy"), a)


def metric_name(c):
    return f"restored 256x256 images/sec @{c['T']} DDIM steps"


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p["bf16_tflops_sustained"], src="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


def sampler_cfg(c):
    import types
    ns = types.SimpleNamespace
    return ns(diffusion=ns(num_diffusion_timesteps=1000), time_travel=ns(T_sampling=c["T"], travel_length=c["tl"], travel_repeat=c["tr"]))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.p, self.path = gpu_index, None, f"/tmp/ddnm_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                      stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], power_w_max=None, samples=0)
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for line in open(self.path):
            f = [s.strip() for s in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), power_w_max=max(pw), samples=len(sm), reasons=sorted(reasons))
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


# torch's CPU conv path collapses when oversubscribed: measured on the B200 host (128 hw threads) one image-forward takes 1.07 s at
# 8 threads, 1.20 s at 16, 1.25 s at 32, 1.92 s at 64 and 51.5 s at 128 (profiles/r01_cpu_threads.txt), so the CPU arms run at the
# thread count where the reference is fastest
def cpu_threads():
    return min(os.cpu_count() or 1, 16)


def cpu_reference_rate(steps, warmup, sample_batch=2, sample_T=3):
    """Reference CPU path for configs[1] on the host cores.  kind "reference": the UNMODIFIED reference code (oracle/_ref: its own
    Model + SuperResolution + ddnm_diffusion, .to('cuda') redirected) on `sample_batch` images with a `sample_T`-step schedule;
    every DDIM step costs the same (one UNet forward + projection + re-noising), so images/sec @100 steps = rate x sample_T / 100.
    Falls back to the oracle port (kind "port") only if oracle/_ref was never built."""
    import torch
    nthreads = cpu_threads()
    T100 = CONFIGS["2"]["T"]
    from oracle import make_ref
    if make_ref.available():
        from oracle import ref_runner
        secs, resid = ref_runner.time_reference_sr4(sample_batch, sample_T, nthreads, repeats=warmup + steps)
        dt = sum(secs[warmup:]) / steps
        kind = "reference"
        what = (f"UNMODIFIED reference (functions/svd_ddnm.py::ddnm_diffusion + guided_diffusion/models.py::Model + "
                f"svd_operators.py::SuperResolution from oracle/_ref, torch CPU fp32), |A x0 - y| = {resid:.1e}")
    else:
        from oracle import operators as O, sampler as S, schedule as SCH, unet_simple as U
        torch.set_num_threads(nthreads)
        cfg = U.SimpleUNetConfig.celeba_hq()
        sd = U.init_state_dict(cfg, 1234)
        op = O.SuperResolution.make(3, RES, 4)
        g = torch.Generator().manual_seed(1234)
        x_orig = torch.rand(sample_batch, 3, RES, RES, generator=g) * 2 - 1
        y = op.A(x_orig.reshape(sample_batch, -1))
        x_T = torch.randn(sample_batch, 3, RES, RES, generator=g)
        betas = SCH.linear_betas()

        def one():
            with torch.no_grad():
                S.ddnm_sample(x_T, lambda a, b: U.forward(sd, a, b, cfg), betas, ETA, op, y,
                              lambda k: torch.randn(sample_batch, 3, RES, RES, generator=g), t_sampling=sample_T)
        for _ in range(warmup):
            one()
        t0 = time.perf_counter()
        for _ in range(steps):
            one()
        dt = (time.perf_counter() - t0) / steps
        kind, what = "port", "oracle port of the reference sampler (oracle/_ref absent), torch CPU fp32"
    rate = sample_batch / (dt / sample_T * T100)
    return rate, dt, dict(cores=nthreads, kind=kind,
                          sample=f"{sample_batch} images x a {sample_T}-step DDNM schedule per bench step ({what}; {nthreads} of {os.cpu_count()} host "
                                 f"threads: more threads are slower), scaled x{T100 / sample_T:.1f} to 100 steps (per-step cost is t-independent)")


def run_reference(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    assert args.config == "2", "the reference arm is defined for configs[1] (celeba sr4)"
    c = CONFIGS["2"]
    steps, warm = max(1, min(args.steps, 3)), min(args.warmup, 1)
    rate, dt, cb = cpu_reference_rate(steps, warm)
    cb["value"], cb["unit"] = rate, UNIT
    line = dict(impl="reference", metric=metric_name(c), value=rate, unit=UNIT, n_gpus=args.gpus, steps=steps, warmup=warm,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="fp32", data="synthetic",
                config=dict(workload=c["workload"], note="CPU path of the reference; bounded sample, see cpu_baseline.sample"),
                cpu_baseline=cb, e2e=dict(value=rate, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


def build_workload(c, dev, precision):
    """(model, operator, plus) of a config on `dev`; weights random-init seed 1234 (no checkpoints offline)."""
    import types
    import numpy as np
    import torch
    from ddnm_b200 import operators as E
    from ddnm_b200.model import Model, create_model
    from ddnm_b200.weights import random_state_dict, random_state_dict_openai
    ns = types.SimpleNamespace
    if c["net"] == "celeba":     # configs/celeba_hq.yml model section
        mcfg = ns(model=ns(type="simple", ch=128, out_ch=3, ch_mult=[1, 1, 2, 2, 4, 4], num_res_blocks=2, attn_resolutions=[16],
                           dropout=0.0, in_channels=3, resamp_with_conv=True),
                  data=ns(image_size=RES), diffusion=ns(num_diffusion_timesteps=1000))
        model = Model(mcfg)
        model.precision = precision
        model.load_state_dict(random_state_dict(mcfg, 1234))
    else:                        # configs/imagenet_256.yml model section
        model = create_model(image_size=256, num_channels=256, num_res_blocks=2, learn_sigma=True, attention_resolutions="32,16,8",
                             num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True, use_fp16=True)
        model.precision = precision
        model.load_state_dict(random_state_dict_openai(model, 1234))
    if c["op"] == "sr4":
        op = E.SuperResolution(3, RES, 4, dev)
    elif c["op"] == "color":
        op = E.Colorization(RES, dev)
    elif c["op"] == "inpaint":   # exp/inp_masks/mask.npy (bits shipped in the fixtures), index construction diffusion.py:466-470
        bits = np.load(os.path.join(ROOT, "tests", "golden", "fullsize.npz"))["mask_bits"]
        mask = torch.from_numpy(np.unpackbits(bits)[: RES * RES].astype(np.int64))
        mr = torch.nonzero(mask == 0).long().reshape(-1) * 3
        op = E.Inpainting(3, RES, torch.cat([mr, mr + 1, mr + 2]), dev)
    elif c["op"] == "deblur":    # diffusion.py:504-509
        sigma = 10
        pdf = lambda z: torch.exp(torch.Tensor([-0.5 * (z / sigma) ** 2]))   # noqa: E731
        k = torch.Tensor([pdf(-2), pdf(-1), pdf(0), pdf(1), pdf(2)])
        op = E.Deblurring((k / k.sum()).to(dev), 3, RES, dev)
    elif c["op"] == "wh":        # diffusion.py:455-459 (global-RNG randperm)
        op = E.WalshHadamardCS(3, RES, 4, torch.randperm(RES ** 2, generator=torch.Generator().manual_seed(1234)).to(dev), dev)
    else:
        raise KeyError(c["op"])
    return model, op, c["sigma_y"] > 0


def main():
    # exactly ONE line on stdout: libraries (NCCL prints its version banner) write to fd 1, so park the real stdout and
    # point fd 1 at stderr until the JSON line is ready
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w")

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ddnm_b200")
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS), help="BASELINE config (2 = configs[1], the driver's line)")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp16"],
                    help="fp32 = fp32-grade 3x fp16 products (parity mode); fp16 = 1 product per MAC, the analogue of use_fp16 (NOT parity grade)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the config's)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed steps of the end-to-end leg (default: --steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-steps", type=int, default=0, help="(ncu runs) skip the e2e / baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args, emit)
    assert args.warmup >= 3 or args.profile_steps, "timing rules: at least 3 warm-up steps"

    import torch
    import torch.distributed as dist
    from ddnm_b200.parallel import shard_rows, sharded_sample
    from ddnm_b200.sampler import ddnm_diffusion, ddnm_plus_diffusion, sample_device
    from ddnm_b200.schedule import time_pairs
    import types

    c = dict(CONFIGS[args.config])
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torchrun)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or c["B"]
    model, op, plus = build_workload(c, dev, args.precision)
    sy = c["sigma_y"]
    conf = sampler_cfg(c)
    betas = torch.from_numpy(__import__("numpy").linspace(1e-4, 2e-2, 1000, dtype="float64")).float().to(dev)
    pairs = time_pairs(1000, c["T"], c["tl"], c["tr"])
    n_pairs, evals = len(pairs), sum(1 for i, j in pairs if j < i)

    # global synthetic batch (identical on every rank), sharded by rows
    Bg = B * world
    g = torch.Generator().manual_seed(1234)
    x_orig = torch.rand(Bg, 3, RES, RES, generator=g) * 2 - 1
    x_T_host = torch.randn(Bg, 3, RES, RES, generator=g).pin_memory()
    lo = rank * B
    y_dev = op.A(x_orig[lo:lo + B].to(dev))
    if plus:
        y_dev = y_dev + sy * torch.randn(y_dev.shape, generator=g).to(dev)
    y_host = y_dev.cpu().pin_memory()
    x_T_dev = x_T_host[lo:lo + B].to(dev)
    torch.manual_seed(1234 + rank)       # per-pair draws differ per rank (independent trajectories)

    def local_fn(xr, yr, nz=None):
        return sample_device(xr, model, betas, ETA, op, yr, sy, plus, conf, noise=nz)

    # ---- untimed: sharded == unsharded on this hardware (SURVEY section 4).  A short schedule over the global batch through
    # parallel.sharded_sample (rows sharded, one all-gather); every rank then recomputes ANOTHER rank's rows itself and compares.
    shard_check = None
    if world > 1:
        cs = dict(c, T=3, tl=1, tr=1)
        conf_s = sampler_cfg(cs)
        gs = torch.Generator().manual_seed(4321)
        xs_g = torch.randn(Bg, 3, RES, RES, generator=gs).to(dev)
        tape = torch.randn(3, Bg, 3, RES, RES, generator=gs).to(dev)
        ys_g = op.A(x_orig.to(dev))
        fn = lambda xr, yr, nz: sample_device(xr, model, betas, ETA, op, yr, 0.0, False, conf_s, noise=nz.contiguous())   # noqa: E731
        full0, _ = sharded_sample(fn, xs_g, ys_g, tape)
        other = (rank + 1) % world
        l2, h2 = shard_rows(Bg, other, world)
        mine, _ = fn(xs_g[l2:h2], ys_g[l2:h2], tape[:, l2:h2])
        diff = torch.tensor([(mine - full0[l2:h2]).abs().max().item()], device=dev)
        dist.all_reduce(diff, op=dist.ReduceOp.MAX)
        shard_check = dict(max_abs_diff=diff.item(), rows=Bg, T_sampling=3,
                           note="parallel.sharded_sample over the global batch vs each rank recomputing the next rank's rows; bit-identical expected")
        del xs_g, tape, ys_g, full0, mine

    def step_device():
        # hot path with x_T / y resident in HBM, draws included (+ the single end-of-run all-gather when N > 1)
        x0, x0p = local_fn(x_T_dev, y_dev)
        if world == 1:
            return x0, x0p
        outs = [torch.empty_like(x0) for _ in range(world)]
        dist.all_gather(outs, x0)
        return outs, x0p

    def step_e2e():
        # public API with HOST buffers: H2D of x_T and y, noise drawn by the API, D2H of both results
        if plus:
            return ddnm_plus_diffusion(x_T_host[lo:lo + B], model, betas, ETA, op, y_host, sy, config=conf)
        return ddnm_diffusion(x_T_host[lo:lo + B], model, betas, ETA, op, y_host, config=conf)

    def timed(fn, steps, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), out

    if args.profile_steps:      # ncu launch list: just run the hot path
        for _ in range(args.profile_steps):
            step_device()
        torch.cuda.synchronize()
        emit(dict(note="profile run, no timing"))
        return

    clocks = ClockSampler(local)
    clocks.start()
    ms_total, (x0, x0p) = timed(step_device, args.steps, args.warmup)
    clk = clocks.stop()
    if args.dump_outputs:
        if world > 1:       # x0 is already every rank's rows; gather the x0 predictions the same way
            x0 = torch.cat(x0)
            parts = [torch.empty_like(x0p) for _ in range(world)]
            dist.all_gather(parts, x0p)
            x0p = torch.cat(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"x0": x0, "x0_pred": x0p})
    del x0, x0p
    e2e_steps = args.e2e_steps or args.steps
    ms_e2e, _ = timed(step_e2e, e2e_steps, 2)
    ms_step = ms_total / args.steps
    value = Bg * 1e3 / ms_step
    e2e_value = Bg * 1e3 / (ms_e2e / e2e_steps)

    if rank == 0:
        info = model.info(B)
        pk = peaks()
        # roofline of the dominant kernel family (the tcgen05 convolution): per-launch CUDA-event timing of one eager forward
        xt = torch.randn(B, 3, RES, RES, device=dev)
        # three eager passes, per launch the fastest: in the regions of short launches the elapsed time between two events measures the
        # host's issue rate rather than the kernel (profiles/r02_attn_anomaly.md), and that jitter is one-sided
        tt = torch.full((B,), 500.0, device=dev)
        prof = model.profile(xt, tt)
        for _ in range(2):
            for a, b in zip(prof, model.profile(xt, tt)):
                a["ms"] = min(a["ms"], b["ms"])
        tc = [p for p in prof if p["kind"] in ("tc", "tcgn")]
        tc_ms, tc_fl = sum(p["ms"] for p in tc), sum(p["flops"] for p in tc)
        all_ms = sum(p["ms"] for p in prof)
        ach = tc_fl / tc_ms / 1e9 if tc_ms > 0 else 0.0
        fwd_launches = sum(4 if p["kind"] == "temb" else (0 if p["kind"] == "memset" else 1) for p in prof)
        traffic = None
        for src in ("r02_conv_traffic.json", "r01_conv_tc_traffic.json"):
            try:   # STATIC: one `ncu --set full` capture of the top launch kept under profiles/ (not re-measured in this run)
                tj = json.load(open(os.path.join(ROOT, "profiles", src)))["top_launch"]
                traffic = dict(bytes=tj["traffic_bytes"], algorithmic_bytes=tj["algorithmic_bytes"], launch=tj["name"],
                               tensor_pipe_active_pct=tj["tensor_pipe_active_pct"],
                               source=f"static: profiles/{src} (ncu --set full capture of this launch, not re-measured by this run)")
                break
            except Exception:
                pass
        terms = 3 if args.precision == "fp32" else 1
        roof = dict(bound="tensor", kernel="conv_tc_kernel / conv_gn_tc_kernel (tcgen05 implicit GEMM, TMA-staged, TMEM accumulators)", achieved=ach,
                    peak=pk["tf_sust"], unit="TFLOP/s", frac=ach / pk["tf_sust"], hw_mma_factor=terms, frac_hw=terms * ach / pk["tf_sust"],
                    peak_source=pk["src"] + ", sustained bf16 cuBLAS", traffic=traffic,
                    launches_per_forward=len(tc), avg_launch_ms=tc_ms / max(1, len(tc)), share_of_forward=tc_ms / all_ms,
                    note=f"achieved = algorithmic conv/GEMM FLOPs (2*M*N*K once) / summed per-launch CUDA-event time; each algorithmic MAC costs {terms} fp16 MMA(s)"
                         + (" (hi*hi+hi*lo+lo*hi) for fp32-grade products, so frac_hw = 3*frac is the tensor-pipe utilisation and 1/3 the ceiling of frac" if terms == 3 else ""))
        line = dict(metric=metric_name(c), value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_step,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="fp32" if args.precision == "fp32" else "fp16", data="synthetic",
                    config=dict(workload=c["workload"], baseline_config=args.config, precision=args.precision, global_batch=Bg,
                                parallelism=f"rows sharded over {world} GPU(s), 1 all-gather at the end",
                                noise="per-pair Gaussian draws inside the timed region (side stream, bounded double buffer)",
                                l2="working set per UNet forward (GiBs of activations) exceeds the 126 MB L2; no flush needed",
                                unet_ms_per_forward=all_ms, unet_evals_per_image=evals, time_pairs=n_pairs,
                                unet_flops_per_image_forward=info["flops_per_forward"] / B, workspace_bytes=info["workspace_bytes"]),
                    clocks=clk, roofline=roof,
                    e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=int(B * 3 * RES * RES * 4 + B * op.y_dim * 4) * world,
                             d2h_bytes_per_step=int(2 * B * 3 * RES * RES * 4) * world, steps=e2e_steps, warmup=2,
                             note="ddnm_b200.sampler.ddnm_diffusion / ddnm_plus_diffusion with pinned host x_T / y, noise drawn inside the call, results returned as CPU tensors"),
                    gpu_launches=int(args.steps * (evals * (fwd_launches + 1 + STEP_KERNELS[c["op"]]) + (n_pairs - evals) + n_pairs)))
        if shard_check is not None:
            line["shard_check"] = shard_check
        if not args.no_cpu_baseline and world == 1 and args.config == "2":
            rate, dt, cb = cpu_reference_rate(1, 0)
            cb["value"], cb["unit"] = rate, UNIT
            line["cpu_baseline"] = cb
        else:
            line["cpu_baseline"] = None
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
