#!/usr/bin/env python
"""bench.py -- shapes/sec of LION's sampling hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

One bench "step" = one full pass of the hot path over one batch: `generate_samples_vada_2prior`
= 1000 denoising steps of the global prior + 1000 of the latent-point prior (PVCNN2-AdaGN)
+ one VAE-decoder pass, for `--batch` shapes of 2048 latent points per GPU (BASELINE.json
configs[1]; at N > 1 every rank samples its own 32 shapes -> weak scaling, and the finished
point clouds are all-gathered once per pass, the path's only collective).  Weights are
key-seeded synthetic tensors (no checkpoints offline), data is synthetic noise.

Printed JSON line (rank 0): the base contract plus
  roofline      the dominant kernel (3x3x3 voxel convolution 64->64 @ 32^3, tcgen05 TF32) timed
                alone with CUDA events via lion_bench_conv; achieved = algorithmic FLOPs / time,
                peak = MEASURED_PEAKS.json bf16 burst / 2 (TF32 runs at half the bf16 rate)
  cpu_baseline  the CPU oracle (oracle/) on the host cores, bounded sample, extrapolated
  e2e           the same pass with all noise supplied from pinned HOST memory (H2D inside the
                timed region) and the point clouds copied back to pinned host memory
  gpu_baseline  (N=1, informational) the UNMODIFIED reference on the same GPU: baseline/ref_gpu_arm.py runs the
                reference's own generate_samples_vada_2prior (copy under baseline/_ref/LION, its JIT-built pvcnn
                kernels, torch cuDNN/cuBLAS) for a FULL 1000+1000-step pass at the same batch, in a child process.
                Falls back to the oracle's eager port (`--impl reference-gpu`) when baseline/_ref is absent.
  parity        (N=1) teacher-forced B=32 parity of one denoising step of both priors against the reference's
                eager path on the GPU (oracle/net.py + the reference's own point kernels), child process
  extra_configs BASELINE configs[3] (CLIP-conditioned prior, B=32, 1 GPU) and, at N=4, configs[2] (64 shapes over
                4 GPUs, 16 per rank): one timed pass each
  per_rank      (N>1) per-rank pass times and the time the sampling stream waited in the all_gather
  env           every LION_* variable that was set (performance knobs); bench refuses to run with any set unless
                --allow-knobs
--impl reference times the reference's own CPU implementation of the path (the oracle port,
restated from the reference and pinned to its goldens) on all host threads.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS = 1000
N_POINTS = 2048
GFLOP_PER_SHAPE = 59.87e3      # SURVEY.md 8d: 1000 x 59.658 + 58.534 + 1000 x 0.154 GFLOP


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu", "parity"])
    ap.add_argument("--batch", type=int, default=32, help="shapes per GPU")
    ap.add_argument("--ddpm-steps", type=int, default=T_STEPS, help="(debug) DDPM steps; the metric is defined at 1000")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--e2e-upload", default="stream", choices=["stream", "first"],
                    help="end-to-end leg: stream the per-step noise upload under the denoising loops, or finish it first")
    ap.add_argument("--e2e-compare", action="store_true", help="(diagnostic) also time the other --e2e-upload mode")
    ap.add_argument("--clock-period-ms", type=int, default=1000, help="nvidia-smi sampling period during the timed region")
    ap.add_argument("--allow-knobs", action="store_true", help="run although LION_* performance knobs are set (they are recorded in the line)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed passes, write what the last one returned as DIR/<name>.npy (float32; rank 0) "
                         "so that two builds can be compared output for output")
    return ap.parse_args()


DUMP_MAX_ELEMS = 4 << 20          # per array: 16 MB of float32, so that a dump stays below 64 MB in all


def dump_outputs(dst, result):
    """Write the 5-tuple returned by generate_samples_vada_2prior as float32 .npy files: the point clouds, the sampled
    latents, their statistics, the NFE count and a fixed sample of the latent-point trajectory (pred_x, T x B x 8192
    floats: the same 4096 positions of every step).  An array larger than DUMP_MAX_ELEMS is replaced by its values at
    a fixed seeded set of flat positions.  The wall-clock sampling time is not an output and is not written."""
    import numpy as np
    import torch
    image, nfe, time_ode_solve, _sampling_time, output = result
    traj = output["eps_list"]["pred_x"]
    n = traj[0].numel()
    pos = torch.from_numpy(np.sort(np.random.RandomState(0).choice(n, min(n, 4096), replace=False))).to(traj[0].device)
    arrays = {"image": image, "nfe": nfe, "time_ode_solve": time_ode_solve, "sampled_eps": output["sampled_eps"],
              "sample_mean_global": output["print/sample_mean_global"], "sample_var_global": output["print/sample_var_global"],
              "pred_x_sample": torch.stack([x.reshape(-1)[pos] for x in traj])}
    os.makedirs(dst, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_MAX_ELEMS:
            a = a.ravel()[np.sort(np.random.RandomState(1).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(dst, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (one looping nvidia-smi process, 1 sample/s by default).
    The query is kept light: at 5 samples/s with power.draw in it, rank 0 -- the only rank that samples -- ran its passes
    2.2 % slower than rank 1 (profiles/r02_bench_n2_final.json: 6666 vs 6519 ms), every query takes the driver lock."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, period_ms=1000):
        self.index = index
        self.period_ms = int(period_ms)
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_models(cfg, device, clip=False):
    import torch
    from lion_b200.models.latent_points_ada_localprior import PVCNN2Prior
    from lion_b200.models.score_sde.resnet import PriorSEDrop, PriorSEClip
    from lion_b200.models.vae_adain import Model
    from tests.synth import synth_state_dict
    shp = lambda m: {k: list(v.shape) for k, v in m.state_dict().items()}
    gp = (PriorSEClip if clip else PriorSEDrop)(cfg.sde, cfg.latent_pts.style_dim, cfg)
    gp.load_state_dict(synth_state_dict(shp(gp), 14))
    lp = PVCNN2Prior(cfg.sde, 1, cfg)
    lp.load_state_dict(synth_state_dict(shp(lp), 11))
    vae = Model(cfg)
    vae.decoder.load_state_dict(synth_state_dict(shp(vae.decoder), 13))
    dae = torch.nn.ModuleList([gp, lp]).to(device).eval()
    return dae, vae.to(device).eval()


# ------------------------------------------------------------------------------------------------
_CPU_STATE = {}


def cpu_threads():
    """oneDNN / OpenMP scale poorly past a few dozen threads on B=1 work and the GPU boxes' 128
    logical cores are shared, so the CPU legs use at most 32 threads (reported as `cores`)."""
    return max(1, min(32, os.cpu_count() or 1))


def cpu_reference_sample(local_steps=1, global_steps=1, batch=1):
    """Bounded sample of the reference's CPU path (oracle port, oracle/net.py): `local_steps`
    PVCNN2Prior denoising steps + `global_steps` global-prior steps at batch `batch`.  The decoder pass
    (58.5 GFLOP, same U-Net minus the time embedding) is costed as one PVCNN2Prior step (59.7 GFLOP).
    Returns (shapes_per_sec extrapolated to 1000 + 1000 + 1 network evaluations, detail)."""
    import torch
    from oracle import net as ON
    from tests.synth import synth_state_dict
    torch.set_num_threads(cpu_threads())
    st = _CPU_STATE.setdefault(batch, {})
    if not st:
        keys = json.load(open(os.path.join(ROOT, "tests", "golden", "keys.json")))
        st["sd_l"], st["sd_g"] = synth_state_dict(keys["prior"], 11), synth_state_dict(keys["global"], 14)
        g = torch.Generator().manual_seed(0)
        st["x"] = torch.randn(batch, 8192, 1, 1, generator=g)
        st["style"] = torch.randn(batch, 128, 1, 1, generator=g)
        st["t"] = torch.full((batch,), 500.0)
        st["spec"] = ON.prior_spec()
    with torch.no_grad():
        t0 = time.perf_counter()
        for _ in range(local_steps):
            ON.prior_forward(st["sd_l"], st["spec"], st["x"], st["t"], st["style"])
        tl = (time.perf_counter() - t0) / local_steps
        t0 = time.perf_counter()
        for _ in range(global_steps):
            ON.global_prior_forward(st["sd_g"], st["style"], st["t"])
        tg = (time.perf_counter() - t0) / global_steps
    total = T_STEPS * (tl + tg) + tl           # seconds per batch (decoder ~ one more local step)
    return batch / total, {"s_per_local_step": tl, "s_per_global_step": tg, "threads": cpu_threads(), "batch": batch}


CPU_SAMPLE = ("%d PVCNN2Prior + %d global-prior denoising step(s) at batch %d on the CPU oracle (port of the reference's PyTorch "
              "path), decoder costed as one PVCNN2Prior step, extrapolated to 1000 + 1000 + 1 evaluations")


def run_gpu_reference(args):
    """--impl reference-gpu (informational, not part of the driver's contract): a GPU port of the
    reference's eager PyTorch path -- oracle/net.py on CUDA tensors (cuDNN / cuBLAS through torch, TF32
    convolutions and cudnn.benchmark as the reference runs them, utils/utils.py:472) with the reference's
    OWN point kernels (oracle/_ref/_pvcnn_backend.so).  The reference's Python modules themselves cannot
    travel to the GPU box.  Bounded sample: a few denoising steps of both priors at batch B, timed with
    CUDA events after a warm-up step, extrapolated to 1000 + 1000 + 1 network evaluations."""
    import torch
    from oracle import diffusion as OD
    from oracle import net as ON
    from oracle import ref_cuda_ops
    from tests.synth import synth_state_dict
    assert torch.cuda.is_available()
    dev = torch.device("cuda", 0)
    torch.backends.cudnn.benchmark = True
    ON.set_point_ops(ref_cuda_ops)
    B = args.batch
    keys = json.load(open(os.path.join(ROOT, "tests", "golden", "keys.json")))
    sd_l = {k: v.to(dev) for k, v in synth_state_dict(keys["prior"], 11).items()}
    sd_g = {k: v.to(dev) for k, v in synth_state_dict(keys["global"], 14).items()}
    spec = ON.prior_spec()
    sched = OD.make_schedule(T_STEPS, 1e-4, 0.02)
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(B, 8192, 1, 1, device=dev, generator=g)
    xg = torch.randn(B, 128, 1, 1, device=dev, generator=g)
    style = torch.randn(B, 128, device=dev, generator=g)
    n_steps = 3

    def local_step(x, t):
        tt = torch.ones(B, device=dev) * (t + 1)
        eps = ON.prior_forward(sd_l, spec, x, tt, style)
        return OD.ddpm_step(sched, x, eps, t, torch.randn(x.shape, device=dev, generator=g))

    def global_step(xg, t):
        tt = torch.ones(B, device=dev) * (t + 1)
        eps = ON.global_prior_forward(sd_g, xg, tt)
        return OD.ddpm_step(sched, xg, eps, t, torch.randn(xg.shape, device=dev, generator=g))

    def timed(step, x0):
        with torch.no_grad():
            x1 = step(x0, T_STEPS - 1)                      # warm-up: cuDNN algorithm search, allocator
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for k in range(n_steps):
                x1 = step(x1, T_STEPS - 2 - k)
            e1.record()
            torch.cuda.synchronize(dev)
            assert torch.isfinite(x1).all()
        return max(e0.elapsed_time(e1) / 1000.0, time.perf_counter() - t0) / n_steps

    tl = timed(local_step, x)
    tg = timed(global_step, xg)
    total = T_STEPS * (tl + tg) + tl                        # seconds per batch of B shapes
    print(json.dumps({"impl": "reference-gpu", "metric": "shapes/sec (1000-step DDPM, 2048 latent pts, B=32)", "value": B / total,
                      "unit": "shapes/s", "n_gpus": 1, "kind": "port: oracle/net.py on CUDA (torch cuDNN/cuBLAS, TF32 convs, eager) + "
                      "the reference's own pvcnn kernels (oracle/_ref)",
                      "sample": "%d + %d denoising steps at batch %d after one warm-up step, extrapolated to 1000 + 1000 + 1 "
                                "network evaluations" % (n_steps, n_steps, B),
                      "detail": {"s_per_local_step": tl, "s_per_global_step": tg}}))



def run_parity(args):
    """--impl parity (child process of the default run; SURVEY.md 8d "parity checks reported with the number"):
    teacher-forced parity AT THE BENCHMARKED BATCH of one denoising step of both priors against the reference's eager
    path on the GPU (oracle/net.py on CUDA tensors = torch cuDNN/cuBLAS + the reference's OWN point kernels from
    oracle/_ref), plus the exactness of the index-producing operators.  The oracle is the checker here, never timed."""
    import torch
    from oracle import net as ON
    from oracle import point_ops, ref_cuda_ops
    from oracle.build_ref import load_ref
    from lion_b200.config import default_prior_cfg
    from lion_b200.models.latent_points_ada_localprior import PVCNN2Prior
    from lion_b200.models.score_sde.resnet import PriorSEDrop
    from lion_b200.third_party.pvcnn import functional as F
    from lion_b200.third_party.pvcnn.functional import furthest_point_sample_indices
    from tests.synth import synth_state_dict
    from tests.util import rel_err, rms_err
    B = args.batch
    dev = torch.device("cuda", 0)
    keys = json.load(open(os.path.join(ROOT, "tests", "golden", "keys.json")))
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, 8192, 1, 1, generator=g)
    style = torch.randn(B, 128, 1, 1, generator=g)
    t = torch.randint(1, 1001, (B,), generator=g).float()
    sd_l, sd_g = synth_state_dict(keys["prior"], 11), synth_state_dict(keys["global"], 14)
    cfg = default_prior_cfg()
    lp = PVCNN2Prior(cfg.sde, 1, cfg); lp.load_state_dict(sd_l)
    gp = PriorSEDrop(cfg.sde, 128, cfg); gp.load_state_dict(sd_g)
    lp, gp = lp.cuda().eval(), gp.cuda().eval()
    eps = lp(x=x.cuda(), t=t.cuda(), condition_input=style.cuda())
    eg = gp(x=style.cuda(), t=t.cuda(), condition_input=None)
    ON.set_point_ops(ref_cuda_ops)
    try:
        with torch.no_grad():
            ref = ON.prior_forward({k: v.to(dev) for k, v in sd_l.items()}, ON.prior_spec(), x.to(dev), t.to(dev), style.to(dev))
            refg = ON.global_prior_forward({k: v.to(dev) for k, v in sd_g.items()}, style.to(dev), t.to(dev))
    finally:
        ON.set_point_ops(point_ops)
    coords = x.view(B, 2048, 4).permute(0, 2, 1)[:, :3].contiguous().cuda()
    nc = coords - coords.mean(2, keepdim=True)
    nc = nc / (nc.norm(dim=1, keepdim=True).max(dim=2, keepdim=True).values * 2.0 + 0.0) + 0.5
    vox_t = torch.round(torch.clamp(nc * 32, 0, 31)).to(torch.int32)
    _, vox = F.voxel_coords(coords, 32)
    rk = load_ref()
    fps_ok = bool(torch.equal(furthest_point_sample_indices(coords, 1024).cpu(), rk.furthest_point_sampling(coords, 1024).cpu()))
    print(json.dumps({"impl": "parity", "batch": B,
                      "against": "reference eager path on the same GPU: oracle/net.py on CUDA (torch cuDNN TF32 convs, cuBLAS) + the reference's own pvcnn kernels (oracle/_ref)",
                      "pvcnn2prior_step": {"max_abs_err_over_max_abs": rel_err(eps, ref), "rms_rel": rms_err(eps, ref), "tolerance": {"max": 1e-2, "rms": 4e-3}},
                      "global_prior_step": {"max_abs_err_over_max_abs": rel_err(eg, refg), "tolerance": {"max": 2e-3}},
                      "voxel_indices_equal_torch_cuda_level0": bool(torch.equal(vox, vox_t)),
                      "fps_indices_equal_reference_kernel_level0": fps_ok,
                      "note": "teacher-forced single step, random timesteps; the free-running 10-step loop is checked against the reference-generated golden in tests (0.2 max / 5e-2 rms: round / arg-max discontinuities amplify 1-ulp differences)"}))


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        v, detail = cpu_reference_sample(1, 1, args.batch)      # the arm's own batch (BASELINE configs[1]: 32 shapes)
        if i >= args.warmup:
            vals.append(v)
    v = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": "shapes/sec (1000-step DDPM, 2048 latent pts, B=32)", "value": v, "unit": "shapes/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * args.batch / v,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "airplane prior, batch %d per GPU, 1000 DDPM steps x (global prior + PVCNN2 latent-point prior) + VAE decoder, 2048 latent pts (BASELINE configs[1])" % args.batch,
                       "global_batch": args.batch,
                       "timed_on": "host CPU, oracle port of the reference's PyTorch path; each step = a bounded sample (1 + 1 denoising steps of the whole batch), extrapolated x1000"},
            "cpu_baseline": {"value": v, "unit": "shapes/s", "cores": cpu_threads(), "kind": "port", "sample": CPU_SAMPLE % (1, 1, args.batch),
                             "detail": detail},
            "e2e": {"value": v, "unit": "shapes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference-gpu":
        run_gpu_reference(args)
        return
    if args.impl == "parity":
        return run_parity(args)
    if args.impl == "reference":
        return run_reference_arm(args)
    knobs = {k: v for k, v in os.environ.items() if k.startswith("LION_")}
    if knobs and not args.allow_knobs:
        sys.exit("bench.py: refusing to run with LION_* knobs set (%s); unset them or pass --allow-knobs "
                 "(they are recorded in the JSON line either way)" % ", ".join(sorted(knobs)))
    import torch
    import torch.distributed as dist
    from lion_b200 import _lib as L
    from lion_b200.config import default_prior_cfg
    from lion_b200.utils.diffusion_pvd import DiffusionDiscretized
    from lion_b200.trainers.train_2prior import generate_samples_vada_2prior

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path for --impl ours)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)
    L.lib()
    B, T = args.batch, args.ddpm_steps
    cfg = default_prior_cfg(num_steps=T)
    dae, vae = build_models(cfg, dev)
    diff = DiffusionDiscretized(cfg.sde, None, cfg)
    shape = vae.latent_shape()
    # the path's single collective: all_gather of the finished clouds, once per pass.  It is issued asynchronously
    # (NCCL's own stream, double-buffered destination) and only waited for before the buffer is reused / at the end
    # of the timed region, so a rank never idles at another rank's pass boundary (round 1 lost 1.7 % to rank skew
    # absorbed there).
    gathered = [[torch.empty(B, N_POINTS, 3, device=dev) for _ in range(world)] for _ in range(2)] if world > 1 else None
    launches = {"n": 0}
    pending = [None, None]
    pass_events = []                                      # (start, end of sampling, end of gather wait) per pass

    def one_pass(seed, record=False):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if record else None
        if record:
            ev[0].record()
        torch.manual_seed(seed * 1000 + rank)             # distinct noise per rank (SURVEY.md 8e)
        result = generate_samples_vada_2prior(shape, dae, diff, vae, B, False)
        img = result[0]
        launches["n"] += L.last_launches(dev)             # decoder pass (the sampling loops count themselves)
        if record:
            ev[1].record()
        if world > 1:
            slot = seed & 1
            if pending[slot] is not None:
                pending[slot].wait()                      # the buffer's previous gather (two passes ago) is done
            pending[slot] = dist.all_gather(gathered[slot], img.contiguous(), async_op=True)
        if record:
            ev[2].record()
            pass_events.append(ev)
        return result

    def drain():
        for i in (0, 1):
            if pending[i] is not None:
                pending[i].wait()
                pending[i] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing: K passes, CUDA events, max over ranks --------------------------
    for i in range(args.warmup):
        one_pass(i)
    drain()
    barrier()
    launches["n"] = 0
    diff.total_gpu_launches = 0
    sampler = ClockSampler(local, args.clock_period_ms)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    last = None
    for i in range(args.steps):
        last = None                                       # the previous pass's 1 GB trajectory goes back to the allocator first
        last = one_pass(100 + i, record=True)
    t_d0 = torch.cuda.Event(enable_timing=True); t_d0.record()
    drain()                                               # every gather has landed: inside the timed region
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = tms.item()
    value = world * B * args.steps / (ms / 1000.0)
    n_launch = launches["n"] + diff.total_gpu_launches
    assert torch.isfinite(last[0]).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)             # before any later pass reuses the sampler's buffers
    del last
    per_rank = None
    if world > 1:
        mine = torch.tensor([[ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])] for ev in pass_events] +
                            [[t_d0.elapsed_time(e1), 0.0]], device=dev)            # [steps+1, 2]
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        if rank == 0:
            import statistics
            samp = [[float(v) for v in r[:-1, 0]] for r in allr]
            tot = [sum(x) for x in samp]
            per_rank = {"pass_ms_per_rank_mean": [round(sum(x) / len(x), 2) for x in samp],
                        "pass_ms_min_median_max_over_ranks": [round(min(map(min, samp)), 2), round(statistics.median([v for x in samp for v in x]), 2),
                                                              round(max(map(max, samp)), 2)],
                        "sampling_ms_total_per_rank": [round(v, 1) for v in tot],
                        "skew_ms_total_max_minus_min": round(max(tot) - min(tot), 2),
                        "allgather_enqueue_ms_per_rank_total": [round(float(r[:-1, 1].sum()), 3) for r in allr],
                        "final_gather_drain_ms_per_rank": [round(float(r[-1, 0]), 3) for r in allr],
                        "note": "the all_gather is asynchronous; ranks only meet in the final drain + barrier"}

    # ---- end to end: all noise from pinned host memory, result back to pinned host --------------
    e2e = None
    if not args.no_e2e:
        g = torch.Generator().manual_seed(1234 + rank)
        hn_g = torch.randn(T + 1, B, 128, 1, 1, generator=g).pin_memory()
        hn_l = torch.randn(T + 1, B, 8192, 1, 1, generator=g).pin_memory()
        hout = torch.empty(B, N_POINTS, 3).pin_memory()
        h2d = (hn_g.numel() + hn_l.numel()) * 4
        d2h = hout.numel() * 4

        # The 1.05 GB of latent-point noise is uploaded in chunks on a copy stream, last timesteps first (the
        # loop consumes z[T-1] .. z[0]); the sampling stream waits only for the chunk it is about to read, so
        # the H2D traffic overlaps the denoising steps instead of preceding them.  Everything stays inside the
        # timed region.
        copy_stream = torch.cuda.Stream(device=dev)
        dl = torch.empty(hn_l.shape, device=dev)
        CH = 50                                                   # timesteps per chunk (13 MB)

        class DeviceNoise:
            """given_noise[1] already on the device: the captured step fetches row t itself (lion_ddpm_fetch_noise)"""

            def __init__(self, block):
                self.device_block = block

            def __getitem__(self, t):
                return self.device_block[t]

        class StreamedNoise:
            """given_noise[1]: z[t] -> device tensor, after making the current stream wait for its upload"""

            def __init__(self):
                self.events = {}
                start = torch.cuda.Event()
                start.record()
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(start)
                    for lo in list(range(1, T + 1, CH))[::-1]:       # rows 1..T hold z[0..T-1]
                        hi = min(T + 1, lo + CH)
                        dl[lo:hi].copy_(hn_l[lo:hi], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(copy_stream)
                        self.events[lo] = ev
                self.waited = set()

            device_block = dl[1:]                                 # row t = z[t]: fetched inside the captured step

            def ensure(self, t):
                lo = 1 + ((t + 1 - 1) // CH) * CH
                if lo not in self.waited:
                    torch.cuda.current_stream().wait_event(self.events[lo])
                    self.waited.add(lo)

            def __getitem__(self, t):
                self.ensure(t)
                return dl[1 + t]

        e2e_ev = []                                               # CUDA events at the phase boundaries of the last pass

        def e2e_pass():
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record()
            dg = hn_g.to(dev, non_blocking=True)
            dl[0].copy_(hn_l[0], non_blocking=True)               # x_T of the latent points
            zl = StreamedNoise()
            if upload_first:
                torch.cuda.current_stream().wait_stream(copy_stream)   # the whole upload precedes the first denoising step
            ev[1].record()
            z_g, _ = diff.run_denoising_diffusion(dae[0], B, shape[0], given_noise=(dg[0], DeviceNoise(dg[1:])))
            ev[2].record()
            z_l, _ = diff.run_denoising_diffusion(dae[1], B, shape[1], condition_input=vae.global2style(z_g),
                                                  given_noise=(dl[0], zl))
            ev[3].record()
            pts = vae.sample(num_samples=B, decomposed_eps=vae.decompose_eps(vae.compose_eps([z_g, z_l])))
            if world > 1:
                dist.all_gather(gathered[0], pts.contiguous())
            hout.copy_(pts, non_blocking=True)
            ev[4].record()
            torch.cuda.synchronize(dev)
            e2e_ev[:] = ev

        def timed_e2e(first):
            nonlocal upload_first
            upload_first = first
            e2e_pass()                                      # warm-up
            barrier()
            t0_ = time.perf_counter()
            for _ in range(n_e2e):
                e2e_pass()
            barrier()
            dt_ = torch.tensor([time.perf_counter() - t0_], device=dev)
            if world > 1:
                dist.all_reduce(dt_, op=dist.ReduceOp.MAX)
            ph = {"h2d_setup": e2e_ev[0].elapsed_time(e2e_ev[1]), "global_prior_loop": e2e_ev[1].elapsed_time(e2e_ev[2]),
                  "local_prior_loop": e2e_ev[2].elapsed_time(e2e_ev[3]), "decoder_gather_d2h": e2e_ev[3].elapsed_time(e2e_ev[4])}
            return dt_, ph

        n_e2e = max(1, min(args.steps, 2))
        upload_first = False
        dt, e2e_phases = timed_e2e(args.e2e_upload == "first")
        e2e_other = None
        if args.e2e_compare:                                # diagnostic: the other upload mode on the same box
            dt_o, ph_o = timed_e2e(args.e2e_upload != "first")
            e2e_other = {"upload": "stream" if args.e2e_upload == "first" else "first",
                         "value": world * B * n_e2e / dt_o.item(), "phases_ms_last_pass": ph_o}
        e2e = {"value": world * B * n_e2e / dt.item(), "unit": "shapes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "note": "x_T and every per-step noise tensor of both priors come from pinned host memory (the 1 GB of latent-point noise streams in 13 MB chunks on a copy stream, overlapped with the denoising steps; each captured step fetches its row of the uploaded block by the device-side step counter); generated points are read back",
               "seconds_per_pass_wall": dt.item() / n_e2e,
               "upload": args.e2e_upload, "phases_ms_last_pass": e2e_phases}
        if e2e_other:
            e2e["other_upload_mode"] = e2e_other

    # ---- phase breakdown (one extra pass, CUDA events; diagnostic only) -------------------------
    phases = None
    if rank == 0 or world == 1:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        torch.manual_seed(4242)
        ev[0].record()
        z_g, _ = diff.run_denoising_diffusion(dae[0], B, shape[0])
        ev[1].record()
        z_l, _ = diff.run_denoising_diffusion(dae[1], B, shape[1], condition_input=vae.global2style(z_g))
        ev[2].record()
        vae.sample(num_samples=B, decomposed_eps=vae.decompose_eps(vae.compose_eps([z_g, z_l])))
        ev[3].record()
        torch.cuda.synchronize(dev)
        phases = {"global_prior_loop_ms": ev[0].elapsed_time(ev[1]), "local_prior_loop_ms": ev[1].elapsed_time(ev[2]),
                  "decoder_ms": ev[2].elapsed_time(ev[3])}
    # ---- the other single-node BASELINE configs: one timed pass each (after a 5-step warm-up run of the same modules)
    extra = {}
    if not args.no_extra_configs and T == T_STEPS:
        def timed_pass(dae_, vae_, diff_, b, clip_feat=None):
            cfg_w = default_prior_cfg(clip=clip_feat is not None, num_steps=5)
            torch.manual_seed(77 + rank)
            generate_samples_vada_2prior(shape, dae_, DiffusionDiscretized(cfg_w.sde, None, cfg_w), vae_, b, False, clip_feat=clip_feat)
            barrier()
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            im, *_ = generate_samples_vada_2prior(shape, dae_, diff_, vae_, b, False, clip_feat=clip_feat)
            if world > 1:
                dist.all_gather([torch.empty_like(im) for _ in range(world)], im.contiguous())
            z.record()
            barrier()
            assert torch.isfinite(im).all()
            tt = torch.tensor([a.elapsed_time(z)], device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return tt.item()
        if world == 1:
            cfg_c = default_prior_cfg(clip=True, num_steps=T)
            dae_c, vae_c = build_models(cfg_c, dev, clip=True)
            cf = torch.randn(B, 512, generator=torch.Generator().manual_seed(7)).to(dev)
            ms_c = timed_pass(dae_c, vae_c, DiffusionDiscretized(cfg_c.sde, None, cfg_c), B, clip_feat=cf)
            extra["configs[3] car prior + CLIP-conditioned AdaGN (PriorSEClip, clip_feat = randn[B,512]), batch %d, 1 GPU" % B] = {
                "value": B / (ms_c / 1000.0), "unit": "shapes/s", "ms_per_pass": ms_c, "passes": 1}
            del dae_c, vae_c
        if world == 4:
            ms_4 = timed_pass(dae, vae, diff, 16)
            extra["configs[2] chair prior, batch 64 over 4 GPUs (16 per rank), 1000 steps"] = {
                "value": 64 / (ms_4 / 1000.0), "unit": "shapes/s", "ms_per_pass": ms_4, "passes": 1,
                "note": "chair / car / airplane priors share one architecture (SURVEY.md 8d); weights are synthetic either way"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (measured alone, CUDA events on its stream) -------------
    import ctypes as C
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    bf16_peak = peaks.get("bf16_tflops", 1590.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops (burst) / 2: kind::tf32 UMMA issues at half the bf16 rate" if peaks \
        else "fallback 1.59 PFLOP/s bf16 (B200_PROFILING.md) / 2"
    ms_k, fl = C.c_float(), C.c_double()
    L.check(L.lib().lion_bench_conv(L.ctx(dev), 27, 64, 64, 32, B, 20, 3, C.byref(ms_k), C.byref(fl), L.stream()), "bench_conv")
    achieved = fl.value / (ms_k.value * 1e-3) / 1e12
    roofline = {"bound": "tensor", "kernel": "lion::tc::k_conv_tc (3x3x3 conv 64->64 @ 32^3, B=%d; the largest dense convolution: 2 launches / denoising step "
                          "since the first convolution of each r=32 PVConv runs in sparse form)" % B,
                "achieved": achieved, "peak": bf16_peak / 2.0, "unit": "TFLOP/s", "frac": achieved / (bf16_peak / 2.0),
                "ms_per_launch": ms_k.value, "flops_per_launch": fl.value, "peak_source": peak_src, "traffic": None}
    try:   # DRAM bytes of the same kernel from the committed ncu --set full capture (B=32 only)
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_conv_fp3_traffic.json")))
        if B == 32:
            roofline["traffic"] = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            roofline["traffic_unit"] = "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum; algorithmic %d)" % tr["algorithmic_bytes"]
    except Exception:
        pass

    cpu = None
    if not args.no_cpu_baseline and world == 1:          # reported on rank 0 at N=1 only
        cpu_reference_sample(1, 1, 4)                    # warm-up (oneDNN primitive creation)
        v, detail = cpu_reference_sample(1, 1, 4)        # 4 shapes: ~20 s of CPU work on the box's cores
        cpu = {"value": v, "unit": "shapes/s", "cores": cpu_threads(), "kind": "port", "sample": CPU_SAMPLE % (1, 1, 4), "detail": detail}

    def child(cmd, timeout):
        """run a helper in a child process (the reference's kernels exit() on a launch error; nothing there may take
        this line down) and parse its last JSON line"""
        try:
            env = {k: v for k, v in os.environ.items() if not k.startswith(("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_", "TORCHELASTIC", "GROUP_"))}
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
            rows = [l for l in r.stdout.splitlines() if l.startswith("{")]
            return json.loads(rows[-1]) if rows else {"unavailable": (r.stderr or "no output")[-400:]}
        except Exception as e:      # noqa: BLE001
            return {"unavailable": repr(e)[:300]}

    # the UNMODIFIED reference on this GPU (full 1000 + 1000 steps at the same batch), else the oracle's eager port
    gpu_ref = None
    if world == 1 and not args.no_gpu_baseline:
        torch.cuda.empty_cache()
        if os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "LION", "models")) and T == T_STEPS:
            gpu_ref = child([sys.executable, os.path.join(ROOT, "baseline", "ref_gpu_arm.py"), "--batch", str(B), "--steps", str(T)], 600)
        if gpu_ref is None or "unavailable" in gpu_ref:
            port = child([sys.executable, os.path.abspath(__file__), "--impl", "reference-gpu", "--batch", str(B)], 200)
            if gpu_ref is not None:
                port["reference_tree_failed"] = gpu_ref["unavailable"]
            gpu_ref = port
    parity = None
    if world == 1 and not args.no_parity:
        torch.cuda.empty_cache()
        parity = child([sys.executable, os.path.abspath(__file__), "--impl", "parity", "--batch", str(B)], 300)

    line = {"metric": "shapes/sec (1000-step DDPM, 2048 latent pts, B=32)", "value": value, "unit": "shapes/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32 (fp32 storage/accumulate)",
            "data": "synthetic",
            "config": {"workload": "airplane prior, batch %d per GPU, %d DDPM steps x (global prior + PVCNN2 latent-point prior) + VAE decoder, 2048 latent pts (BASELINE configs[1])" % (B, T),
                       "global_batch": B * world, "parallelism": "dp%d (independent shapes, one all_gather per pass)" % world,
                       "l2": "per-step working set (303 MB voxel grids) exceeds the 126 MB L2; no flush needed",
                       "weights": "key-seeded synthetic (tests/synth.py)"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": n_launch,
            "ms_per_denoise_step_pair": ms / args.steps / T,
            "tensor_roofline_frac_whole_job": (value * GFLOP_PER_SHAPE / 1e3 / world / (bf16_peak / 2.0)) if T == T_STEPS else None,
            "phases": phases, "roofline": roofline, "cpu_baseline": cpu, "gpu_baseline": gpu_ref, "parity": parity,
            "extra_configs": extra, "per_rank": per_rank, "env": knobs}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
