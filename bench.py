#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: iterations/sec of pixray's per-iteration hot path, synthetic seeded weights and
prompts.  Default = "vqgan imagenet_f16_16384 256x256, ViT-B/16, cutn=64" (configs[1], the configuration the metric is
quoted on); --config 3 | 4 | 5 selects the other BASELINE configurations.

    python bench.py --gpus 1 --steps K --warmup W             engine arm (this repo's CUDA engine)
    python bench.py --impl reference --gpus N --steps K ...    reference arm: the reference's PyTorch path on the host
                                                               cores (oracle/ref_path.py driving torch CPU ops)
    python bench.py ... --dump-outputs DIR                     also write the last timed step's z and losses as DIR/*.npy

One "step" = one train() iteration (pixray.py:1436-1512): synth -> MakeCutouts -> encode_image -> Prompt losses ->
backward -> Adam -> clip_z.  Prints ONE JSON line on rank 0.
  value : device-resident loop through the C ABI (pxr_iterate), CUDA events on the engine stream, max over ranks
  e2e   : the same iterations through the public module API (pixray_b200.api.do_init + api.train, what pixray.run()
          executes), host-resident parameters in, the loss record out every step
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CUT_SIZE = 224
# BASELINE.json configs[1..4]; lr: pixray.py:1745 default learning_rate (fft: fftdrawer.py:21; vdiff: set per iteration)
CONFIGS = {
    2: dict(metric="iters/sec @ 256^2 VQGAN, ViT-B/16, cutn=64",
            workload="vqgan imagenet_f16_16384 256x256, ViT-B/16, cutn=64 (BASELINE.json configs[1])",
            drawer="vqgan", image=(256, 256), clips=["ViT-B/16"], cutn=64, lr=0.2, shard=True),
    3: dict(metric="iters/sec @ 512^2 VQGAN, ViT-B/16 + ViT-B/32, cutn=128",
            workload="vqgan imagenet_f16_16384 512x512, ViT-B/16 + ViT-B/32, cutn=128 (BASELINE.json configs[2])",
            drawer="vqgan", image=(512, 512), clips=["ViT-B/16", "ViT-B/32"], cutn=128, lr=0.2, shard=True),
    4: dict(metric="iters/sec @ 256^2 vdiff cc12m_1, ViT-B/16, cutn=64",
            workload="vdiff cc12m_1 256x256, ViT-B/16, cutn=64 (BASELINE.json configs[3])",
            drawer="vdiff", image=(256, 256), clips=["ViT-B/16"], cutn=64, lr=0.01, shard=True),
    5: dict(metric="iters/sec @ 512^2 fft drawer, ViT-L/14, cutn=256",
            workload="fft 512x512, ViT-L/14, cutn=256, one prompt per GPU (BASELINE.json configs[4])",
            drawer="fft", image=(512, 512), clips=["ViT-L/14"], cutn=256, lr=0.3, shard=False),
}


def config_dict(cfg, world, shard, extra=None):
    """The `config` object: IDENTICAL keys in the engine arm and the reference arm."""
    d = {"workload": cfg["workload"], "cutn": cfg["cutn"], "image": "%dx%d" % cfg["image"], "clip": " + ".join(cfg["clips"]),
         "drawer": cfg["drawer"], "weights": "seeded random (no checkpoints offline)",
         "parallelism": (f"one problem, {cfg['cutn']} cutouts sharded over {world} rank(s) ({cfg['cutn'] // max(world, 1)} each), "
                         "drawer replicated" if shard else f"{world} independent replica(s), one problem per GPU"),
         "l2": "per-step working set (saved activations, GBs) >> 126 MB L2, no explicit flush"}
    if extra:
        d.update(extra)
    return d


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tflops_burst=p["bf16_tflops"], tflops_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm, reasons, smax = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                smax = float(s[1])
                for nm, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=smax, reasons=sorted(reasons),
                    samples=len(sm))


def drawer_state_dict(cfg, seed=0):
    from pixray_b200 import synthetic as S
    from pixray_b200.engine import VQGAN_F16_16384
    if cfg["drawer"] == "vqgan":
        return S.vqgan_state_dict(VQGAN_F16_16384, seed)
    if cfg["drawer"] == "vdiff":
        return S.vdiff_state_dict(seed)
    return None


def algorithmic_flops(cfg):
    """fwd + dgrad-only bwd = 2 x fwd (SURVEY.md 8d)."""
    from pixray_b200 import synthetic as S
    from pixray_b200.engine import CLIP_ARCH, VQGAN_F16_16384
    fl = sum(cfg["cutn"] * S.vit_fwd_flops(CLIP_ARCH[m]) for m in cfg["clips"])
    if cfg["drawer"] == "vqgan":
        fl += S.vqgan_decoder_fwd_flops(VQGAN_F16_16384, cfg["image"])
    elif cfg["drawer"] == "vdiff":
        fl += 831.5e9 * (cfg["image"][0] * cfg["image"][1]) / (256 * 256)
    return 2 * fl


# ---------------------------------------------------------------------------------------------- reference / CPU arm
def effective_cores():
    """Threads the process can really use: affinity mask and cgroup CPU quota, not the host's core count."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        pass
    return max(1, n)


def pick_threads():
    """torch fp32 GEMM throughput probe over a few thread counts (oversubscribed boxes get slower with more)."""
    n = effective_cores()
    cands = sorted({n, max(1, n // 2), min(n, 64), min(n, 32), min(n, 16), min(n, 8)}, reverse=True)
    a, b = torch.randn(1024, 1024), torch.randn(1024, 1024)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.perf_counter()
        for _ in range(8):
            a @ b
        dt = time.perf_counter() - t0
        if dt < best_t * 0.9:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


class CpuReference:
    """The reference's per-iteration body on host cores: the oracle restatement of pixray.train() (torch fp32 CPU ops)."""

    def __init__(self, cfg, seed=0):
        from oracle import ref_path as R
        from pixray_b200 import synthetic as S
        from pixray_b200.cutouts import sample_transforms
        from pixray_b200.engine import CLIP_ARCH
        self.R, self.cfg = R, cfg
        self.clips, self.prompts = [], []
        for i, m in enumerate(cfg["clips"]):
            a = CLIP_ARCH[m]
            clip = R.ClipVisual(224, a["patch"], a["width"], a["layers"], a["heads"], a["out_dim"])
            clip.load_state_dict(S.clip_state_dict(a, seed + 1 + i))
            self.clips.append(clip.eval().requires_grad_(False))
            self.prompts.append(S.prompts(a["out_dim"], (1.0, 0.1), seed + 2 + i))
        H, W = cfg["image"]
        if cfg["drawer"] == "vqgan":
            sd = drawer_state_dict(cfg, seed)
            vq = R.VQModel()
            vq.load_state_dict(sd)
            vq.eval().requires_grad_(False)
            self.z = S.z0_vqgan(sd["quantize.embedding.weight"], (H // 16, W // 16), seed + 3)
            self.synth = lambda z, it: R.vqgan_synth(vq, z)
            zmin, zmax = R.vqgan_z_bounds(vq)
            self.clip_z = lambda z: torch.maximum(torch.minimum(z, zmax), zmin)
        elif cfg["drawer"] == "fft":
            self.z = (0.01 * torch.randn(1, 3, H, W // 2 + 1, 2, generator=torch.Generator().manual_seed(seed))).contiguous()
            self.synth = lambda z, it: R.fft_synth(z)
            self.clip_z = lambda z: z
        else:  # vdiff
            from pixray_b200.util import vdiff_schedule
            model = R.VDiffCC12M1()
            ref_sd = drawer_state_dict(cfg, seed)
            with torch.no_grad():
                model.map_ff.copy_(ref_sd["mapping_timestep_embed.weight"])
                model.t_ff.copy_(ref_sd["timestep_embed.weight"])
                for key, m in model.keys:
                    for n, prm in m.named_parameters():
                        prm.copy_(ref_sd[f"{key}.{n}"])
            model.eval().requires_grad_(False)
            self.sched = vdiff_schedule(1000)
            ce = self.prompts[0][0][0]
            self.z = (torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(seed)) * float(self.sched[2][0])).contiguous()
            st, al, sg = self.sched
            self.synth = lambda z, it: R.vdiff_synth(model, z, torch.tensor([float(st[it])]), ce, float(al[it]), float(sg[it]))[0]
            self.clip_z = lambda z: z
        self.T = torch.from_numpy(sample_transforms(cfg["cutn"], CUT_SIZE, seed))
        self.adam = R.AdamState(self.z)

    def iteration(self, cutn_sample, it):
        """Returns (seconds in the drawer forward + backward + optimiser, seconds in MakeCutouts + CLIP on cutn_sample cutouts)."""
        from pixray_b200.cutouts import sample_color_jitter
        R, cfg = self.R, self.cfg
        t0 = time.perf_counter()
        zz = self.z.detach().clone().requires_grad_(True)
        out = self.synth(zz, it)
        t1 = time.perf_counter()
        g = torch.Generator().manual_seed(it)
        facs = torch.rand(cutn_sample, generator=g) * 0.1
        noise = torch.randn(cutn_sample, 3, CUT_SIZE, CUT_SIZE, generator=g)
        out_d = out.detach().requires_grad_(True)
        jit = torch.from_numpy(sample_color_jitter(cfg["cutn"], 2000 + it)[:cutn_sample])  # K.ColorJitter rows (pixray.py:416, 436)
        batch = R.make_cutouts(out_d, self.T[:cutn_sample], CUT_SIZE, "reflection" if it % 2 == 0 else "border", 0.5, facs,
                               noise, cutn_zoom=int(0.6 * cutn_sample), jitter=jit)
        loss = 0.0
        for clip, pms in zip(self.clips, self.prompts):
            emb = R.encode_image(clip, batch).float()
            loss = loss + sum(R.prompt_loss(emb, *p) for p in pms)
        loss.backward()
        t2 = time.perf_counter()
        out.backward(out_d.grad)
        self.z = self.clip_z(self.adam.step(self.z, zz.grad, cfg["lr"]))
        t3 = time.perf_counter()
        return (t1 - t0) + (t3 - t2), (t2 - t1)


def run_cpu_reference(cfg, steps, budget_s, seed=0):
    """Times `steps_run` (<= steps) iterations of the reference path, each on the FULL cutn when one such iteration fits the
    budget a few times over; otherwise on a cutout subset, reported as measured, with the extrapolation to the full cutn
    in separate fields.  No hidden scaling: ms_per_step is the measured time of the steps that ran."""
    cores = pick_threads()
    ref = CpuReference(cfg, seed)
    cutn = cfg["cutn"]
    td, tc = ref.iteration(min(4, cutn), 0)  # calibration (also the warm-up of the thread pool / allocator)
    per_cut = tc / min(4, cutn)
    full = td + per_cut * cutn
    if full * 2 <= budget_s:
        cutn_sample = cutn
    else:
        cutn_sample = cutn
        while cutn_sample > 4 and (td + per_cut * cutn_sample) * 2 > budget_s:
            cutn_sample //= 2
    steps_run = int(max(1, min(steps, budget_s // max(td + per_cut * cutn_sample, 1e-9))))
    tds, tcs = [], []
    for it in range(1, 1 + steps_run):
        a, b = ref.iteration(cutn_sample, it)
        tds.append(a)
        tcs.append(b)
    t_meas = float(np.mean(tds)) + float(np.mean(tcs))
    t_full = float(np.mean(tds)) + float(np.mean(tcs)) * (cutn / cutn_sample)
    sample = (f"{steps_run} step(s) of: full drawer synth fwd+bwd + Adam/clip_z, MakeCutouts (ColorJitter incl.) + CLIP fwd+bwd on "
              f"{cutn_sample} of {cutn} cutouts; torch fp32, {cores} threads")
    out = dict(value=1.0 / t_full, unit="iters/sec", cores=cores, kind="port", sample=sample, ms_per_step=t_meas * 1e3,
               steps_run=steps_run, cutn_timed=cutn_sample)
    if cutn_sample != cutn:
        out["extrapolation"] = {"from_cutn": cutn_sample, "to_cutn": cutn, "cutout_part_scale": cutn / cutn_sample,
                                "measured_ms_per_step": t_meas * 1e3, "full_ms_per_step": t_full * 1e3,
                                "note": "value = 1 / full_ms_per_step; the cutout + CLIP part is linear in the cutout count"}
    return out


# ---------------------------------------------------------------------------------------------- engine arm
def run_engine(args, cfg, rank, world):
    import torch.distributed as dist
    from pixray_b200 import api
    from pixray_b200 import engine as E
    from pixray_b200 import synthetic as S
    from pixray_b200.util import vdiff_schedule
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # multi-GPU (DESIGN.md, row e).  "shard" (default where the config shards): ONE optimisation problem, the cutouts
    # split over the ranks, drawer replicated, NCCL on {min, max}, the range-gradient sums and the image gradient: strong
    # scaling.  "replicas": N independent problems, no collective: weak scaling (config 5, or --parallel replicas).
    shard = cfg["shard"] and args.parallel == "shard"
    kind = {"vqgan": E.DRAWER_VQGAN, "vdiff": E.DRAWER_VDIFF, "fft": E.DRAWER_FFT}[cfg["drawer"]]
    cutn, image, lr = cfg["cutn"], cfg["image"], cfg["lr"]
    clip_cfgs = [E.CLIP_ARCH[m] for m in cfg["clips"]]
    if shard:
        eng = E.B200Engine(drawer=kind, image_hw=image, cutn=cutn, clip=clip_cfgs, noise_fac=0.1, seed=0, device=local_rank,
                           rank=rank, world=world)
    else:
        eng = E.B200Engine(drawer=kind, image_hw=image, cutn=cutn, clip=clip_cfgs, noise_fac=0.1, seed=rank, device=local_rank)
    sd = drawer_state_dict(cfg, 0)
    if sd is not None:
        eng.load_module(E.MOD_VQGAN, sd)
    for i, a in enumerate(clip_cfgs):
        eng.load_module(E.MOD_CLIP0 + i, S.clip_state_dict(a, 1 + i))
    eng.finalize()
    if shard and world > 1:
        eng.init_comm()
    jobs = 1 if shard else world
    all_prompts = []
    for i, a in enumerate(clip_cfgs):
        pr = S.prompts(a["out_dim"], (1.0, 0.1), 2 + i)
        all_prompts.append(pr)
        eng.set_prompts(i, torch.cat([p[0] for p in pr]).numpy(), [p[1] for p in pr], [p[2] for p in pr])
    total = args.warmup + args.steps + 2
    if kind == E.DRAWER_VQGAN:
        z = S.z0_vqgan(sd["quantize.embedding.weight"], (image[0] // 16, image[1] // 16), 3).cuda()
    elif kind == E.DRAWER_FFT:
        z = (0.01 * torch.randn(eng.z_shape, device="cuda")).contiguous()
    else:
        st_, al_, sg_ = vdiff_schedule(total)
        eng.vdiff_set_schedule(st_, al_, sg_)
        eng.vdiff_set_clip_embed(all_prompts[0][0][0].numpy())
        z = (torch.randn(eng.z_shape) * float(sg_[0])).cuda().contiguous()
        vd_noise = torch.randn(eng.z_shape, device="cuda")
    ext = torch.cuda.ExternalStream(eng.stream_ptr())

    def step(it):
        if kind == E.DRAWER_VDIFF:  # pixray.py:1489-1495: fresh Adam at the schedule's rate, then makenoise
            eng.reset_optimizer()
            eng.iterate(z, min(float(sg_[it] / al_[it]) * 0.001, 0.01), it)
            eng.lib.pxr_vdiff_renoise(eng.h, eng._p_inplace(z, "z"), it, eng._p(vd_noise))
        else:
            eng.iterate(z, lr, it)

    def barrier():
        eng.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- device-resident arm: engine RNG for the cutouts, no host traffic inside the timed region
    for it in range(args.warmup):
        step(it)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    n0 = eng.num_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for it in range(args.warmup, args.warmup + args.steps):
        step(it)
    e1.record(ext)
    barrier()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    launches = eng.num_launches() - n0
    if args.dump_outputs and rank == 0:  # before profile_iteration, which steps z once more
        dump_outputs(args.dump_outputs, z=z, losses=eng.read_losses())
    # ---- per-kernel split for the roofline of the dominant kernel family
    prof = eng.profile_iteration(z, lr, args.warmup + args.steps)
    barrier()
    eng.close()
    del eng
    torch.cuda.empty_cache()

    # ---- e2e arm: the public module API -- what pixray.run() executes: api.do_init once, then api.train per step.  Every
    # step stages that iteration's cutout parameters host -> device from pinned memory (engine-owned ring) and the step's
    # loss record comes back device -> host (pinned status record written by the optimiser kernel; the host polls it)
    api.reset_settings()
    size = [image[1], image[0]]
    api.add_settings(prompts="a synthetic prompt|a second prompt:0.1", drawer={"vqgan": "vqgan", "vdiff": "vdiff", "fft": "fft"}[cfg["drawer"]],
                     size=size, clip_models=",".join(cfg["clips"]), num_cuts=cutn, iterations=total + 3, batches=1,
                     vector_prompts="none", b200_allow_synthetic=True, seed="0", learning_rate_drops=[], outdir="",
                     learning_rate=lr, cuda_device=f"cuda:{local_rank}", save_every=10 ** 9, display_every=10 ** 9,
                     b200_rank=rank if shard else 0, b200_world=world if shard else 1)
    settings = api.apply_settings()
    api.do_init(settings)
    st = api._state
    ext2 = torch.cuda.ExternalStream(st.engine.stream_ptr())
    it_api = 0
    for _ in range(min(3, args.warmup)):
        api.train(settings, it_api)
        it_api += 1
    st.engine.sync()
    if world > 1:
        dist.barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    f0.record(ext2)
    for _ in range(args.steps):
        api.train(settings, it_api)
        it_api += 1
    f1.record(ext2)
    st.engine.sync()
    wall_e2e = (time.perf_counter() - w0) * 1e3
    ms_e2e = max(f0.elapsed_time(f1), 0.0)
    if ms_e2e < 0.5 * wall_e2e:  # host-paced loop (per-step synchronisation): the wall clock is the honest figure
        ms_e2e = wall_e2e
    rec = st.engine.poll_status() if getattr(st, "managed", False) else None
    last_losses = rec["losses"].tolist() if rec is not None else (None if st.losses is None else np.asarray(st.losses).tolist())
    n_local = cutn // (world if shard else 1)
    h2d = n_local * 12 * 4  # homographies (9) + ColorJitter rows (3) per local cutout, pinned ring -> device
    d2h = 296 if getattr(st, "managed", False) else 64 * 4
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    clocks = sampler.summary()
    # DRAM bytes per tensor-core launch from the committed ncu pass over one iteration (not measurable live without a profiler)
    traffic, traffic_src = None, None
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp) and world == 1 and args.config == 2:
            with open(tp) as f:
                tj = json.load(f)
            traffic, traffic_src = tj["gemm_dram_bytes_per_launch"], tj["source"]
            break
    S_flops = algorithmic_flops(cfg)
    gemm_tflops = prof["gemm_flops"] / (prof["gemm_ms"] * 1e-3) / 1e12 if prof["gemm_ms"] > 0 else 0.0
    nl = max(1, prof["gemm_launches"])
    line = {
        "metric": cfg["metric"], "value": jobs * args.steps / (ms * 1e-3), "unit": "iters/sec", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if shard else "weak", "vs_baseline": None, "dtype": "f16 operands, f32 accumulate",
        "data": "synthetic",
        "config": config_dict(cfg, world, shard, {"algorithmic_flops_per_iter": S_flops, "bench_config": args.config,
                                                  "collectives": ("NCCL allreduce: {min,max} fwd, range-gradient sums + image gradient + losses bwd"
                                                                  if shard and world > 1 else "none")}),
        "clocks": clocks,
        "e2e": {"value": jobs * args.steps / (ms_e2e * 1e-3), "unit": "iters/sec", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "through": "pixray_b200.api.do_init + api.train (the loop of pixray.run())",
                "host_sync_per_step": not getattr(st, "managed", False), "last_losses": last_losses},
        "gpu_launches": launches,
        "roofline": {"kernel": "tcgen05 family: gemm_tc*/gemm_tce* (GEMM / implicit-GEMM conv) + attn_fwd/attn_bwd (fused attention)", "bound": "tensor",
                     "achieved": gemm_tflops, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / peaks["tflops_sustained"], "traffic": traffic,
                     "traffic_unit": "bytes/launch (dram read+write)", "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": prof.get("gemm_bytes", 0.0) / nl,
                     "peak_source": peaks["source"] + ", sustained bf16/f16 GEMM figure",
                     "launches_per_iter": prof["gemm_launches"], "gemm_ms_per_iter": prof["gemm_ms"],
                     "other_ms_per_iter": prof["other_ms"], "iter_ms_profiled": prof["total_ms"],
                     "algorithmic_flops_per_launch": prof["gemm_flops"] / nl,
                     # FLOPs the tensor-core launches of one iteration actually execute (sum of 2 M N K over the plans).
                     # Below config.algorithmic_flops_per_iter -- the full model on every row, what the reference's
                     # PyTorch path computes -- by the dead rows of the last ViT layer (only the class token's row of
                     # each image reaches the embedding; DESIGN.md 4).  whole_iter_tflops uses the EXECUTED count.
                     "executed_flops_per_iter": prof["gemm_flops"],
                     "whole_iter_tflops": min(S_flops, prof["gemm_flops"]) * args.steps / (ms * 1e-3) / 1e12},
    }
    if not args.no_cpu_baseline:
        r = run_cpu_reference(cfg, steps=1, budget_s=25.0)
        line["cpu_baseline"] = {k: r[k] for k in r if k in ("value", "unit", "cores", "kind", "sample", "extrapolation")}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: what a caller of the timed path holds after its last step (z, updated in place, and the loss vector
    of that step), one float32 DIR/<name>.npy each.  z is at most a few MB in every config, so it is written whole.
    Measured on a B200: two runs of config 2 give identical bits; configs 4 (vdiff) and 5 (fft) do not, on identical inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32))


_JSON_FD = None


def emit(line):
    """The ONE stdout line of the contract.  Library banners written to fd 1 while the job runs (NCCL prints its version
    there) are diverted to stderr by main(); the JSON goes to the real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configuration (default 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parallel", default="shard", choices=["shard", "replicas"],
                    help="N > 1: shard the cutouts of one problem over the ranks (default) or run N independent replicas")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's outputs (z, losses) as DIR/<name>.npy; the "
                         "inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs dumps the engine arm's timed path")
    if args.warmup < 3:
        args.warmup = 3
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        if rank != 0:
            return
        shard = cfg["shard"] and args.parallel == "shard"
        r = run_cpu_reference(cfg, args.steps, budget_s=150.0)
        line = {"impl": "reference", "metric": cfg["metric"], "value": r["value"], "unit": "iters/sec", "n_gpus": args.gpus,
                "steps": r["steps_run"], "steps_requested": args.steps, "warmup": 1, "warmup_requested": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "strong" if shard else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(cfg, args.gpus, shard, {"algorithmic_flops_per_iter": algorithmic_flops(cfg), "bench_config": args.config,
                                                              "collectives": "none (host cores, one process)"}),
                "cpu_baseline": {k: r[k] for k in r if k in ("value", "unit", "cores", "kind", "sample", "extrapolation")},
                "e2e": {"value": r["value"], "unit": "iters/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0,
                "note": ("ms_per_step is the MEASURED time of the steps that ran (steps = how many ran inside the time budget, "
                         "warmup = the one calibration step); `value` equals 1000 / ms_per_step unless `cpu_baseline.extrapolation` "
                         "is present")}
        emit(line)
        return
    run_engine(args, cfg, rank, world)


if __name__ == "__main__":
    main()
