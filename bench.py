#!/usr/bin/env python
"""bench.py -- poses/s of the SAM-6D pose-estimation matching path on B200 (BASELINE.json config #2).

A step = one pass of the hot path (Net.forward after the RGB backbone: FPS, geometric embedding, coarse and fine
sparse-to-dense point matching, pose solvers) over one batch of 32 synthetic proposals x 2048 scene points x 2048 template
points, 256-d features, 1024 CAD samples.  Under torchrun every rank runs the same per-GPU batch (weak scaling, proposals
sharded, no data-path collective) and the step ends with the one all-gather of final poses.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm
  python bench.py ... --dump-outputs DIR                        our arm, and the poses of its last timed step as DIR/*.npy
  python bench.py --impl reference ...                          the reference algorithm on the host cores (oracle port)
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = "pem_matching_32x2048x2048"
B_PER_GPU, N_PTS, N_MODEL, C_FEAT = 32, 2048, 1024, 256
METRIC, UNIT = "poses/sec", "poses/s"
REF_ARM_B = 1
CPU_SAMPLE_B = 8
DUMP_LIMIT_BYTES = 64 << 20


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tensor=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, tensor=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML when it is importable (a query
    takes ~1 ms, so a 100 ms timed region still gets tens of samples), else the nvidia-smi command line every 0.2 s."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            dev = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = int(dev.split(",")[index]) if dev and all(x.strip().isdigit() for x in dev.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _nvml_sample(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        bits = [0x8, 0x40, 0x20, 0x4]          # HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap
        return [str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits]

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.samples.append(self._nvml_sample())
                    time.sleep(0.005)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unsampled"])
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                    reasons=reasons, samples=len(self.samples), source="nvml" if self.nvml is not None else "nvidia-smi")


def host_threads() -> int:
    """cores this process may really use: the smaller of the affinity mask and the cgroup CPU quota (os.cpu_count() reports the
    machine, and oversubscribing torch's intra-op pool beyond the quota makes the CPU legs several times slower)"""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, quota // period))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def dump_outputs(out_dir: str, arrays: dict, limit_bytes: int = DUMP_LIMIT_BYTES):
    """write every array as out_dir/<name>.npy in float32.  Above limit_bytes in all, the same fixed, seeded sample of
    proposals (rows along the first axis, kept in order) is written for every array."""
    arrays = {k: v.detach().to(torch.float32).cpu() for k, v in arrays.items()}
    rows = next(iter(arrays.values())).shape[0]
    per_row = sum(v[0].numel() * 4 for v in arrays.values()) if rows else 0
    if rows * per_row > limit_bytes:
        keep = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:limit_bytes // per_row].sort()[0]
        arrays = {k: v[keep] for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.numpy())


def cpu_oracle_throughput(reps: int, threads: int, nprop: int = 0):
    """the reference algorithm (oracle port, torch fp32 on the host) on a bounded sample of the workload"""
    from oracle import pem_oracle as po
    nprop = nprop or CPU_SAMPLE_B
    torch.set_num_threads(threads)
    sd = po.make_state_dict(seed=1)
    inp = po.make_inputs(B=nprop, n=N_PTS, n_model=N_MODEL, seed=1)
    torch.manual_seed(1)
    rand = torch.rand(nprop, po.N_PROPOSAL1 * 3)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        po.pem_forward(sd, inp["pts"], inp["dense_fm"], inp["dense_po"], inp["dense_fo"], inp["model"], rand=rand)
        times.append(time.perf_counter() - t0)
    return nprop / (sum(times) / len(times)), times


def same_box_reference(dev, B):
    """SURVEY.md 8(d) / 2.3: the reference formulation on the SAME B200 -- (i) the reference algorithm (oracle port: the
    reference's own torch ops) on .cuda() with the reference's own pointnet2 CUDA kernels (oracle/_ref) underneath, as
    `ref_gpu_poses_per_s`; (ii) the reference `_ext` FPS / ball-query kernels timed next to ours on the bench shapes.
    Checker / baseline code only: nothing here is on the product path."""
    out = {}
    try:
        from oracle import pem_oracle as po, pn2
        from sam6d_b200 import ops
        ref = pn2._ref()
        x = po.make_inputs(B=B, n=N_PTS, n_model=N_MODEL, seed=1)["dense_po"].to(dev)
        x2 = torch.cat([x, x.flip(1)], dim=0).contiguous()                      # 2B clouds, the launch shape of the step
        x2 = (x2 / (x2.norm(dim=2).amax(dim=1).reshape(-1, 1, 1) + 1e-6)).contiguous()   # unit radius, as Net.forward feeds them

        def t_us(fn, reps=5):
            fn(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record(); torch.cuda.synchronize()
            return 1e3 * e0.elapsed_time(e1) / reps
        out["fps_2048_to_196_us"] = dict(clouds=2 * B, reference_ext=t_us(lambda: ref.furthest_point_sampling(x2, 196)),
                                         ours=t_us(lambda: ops.furthest_point_sampling(x2, 196)))
        out["ball_query_r0.1x32_r0.2x64_us"] = dict(
            clouds=2 * B, reference_ext=t_us(lambda: (ref.ball_query(x2, x2, 0.1, 32), ref.ball_query(x2, x2, 0.2, 64))),
            ours=t_us(lambda: ops.ball_query_pair(x2, x2, 0.1, 32, 0.2, 64)))
        sd = {k: v.to(dev) for k, v in po.make_state_dict(seed=1).items()}
        inp = {k: v.to(dev) for k, v in po.make_inputs(B=B, n=N_PTS, n_model=N_MODEL, seed=1).items()}
        torch.manual_seed(1)
        rand = torch.rand(B, po.N_PROPOSAL1 * 3, device=dev)
        run = lambda: po.pem_forward(sd, inp["pts"], inp["dense_fm"], inp["dense_po"], inp["dense_fo"], inp["model"], rand=rand)  # noqa: E731
        with torch.no_grad():
            us = t_us(run, reps=2)
        out["ref_gpu_poses_per_s"] = B / (us * 1e-6)
        out["ref_gpu_ms_per_step"] = us * 1e-3
        out["ref_gpu_note"] = ("reference algorithm (oracle port = the reference's torch ops, fp32, stock cuBLAS / cuSOLVER / eager kernels of "
                               f"torch {torch.__version__}) + the reference's own pointnet2 CUDA kernels, {B} proposals per step on this GPU")
    except Exception as e:                                                        # reported, never fatal for the bench line
        out["unavailable"] = f"{type(e).__name__}: {e}"[:300]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    # The step's sample is sized from a 1-proposal warm-up so that K steps end within a few minutes: 4 proposals per step
    # (better host throughput per pose) when that fits ~4 minutes, otherwise 1.
    t0 = time.perf_counter()
    cpu_oracle_throughput(1, threads, 1)
    t1 = time.perf_counter() - t0
    nprop = 4 if t1 * 2.5 * max(1, args.steps) < 240.0 else 1
    t0 = time.perf_counter()
    val, times = cpu_oracle_throughput(max(1, args.steps), threads, nprop)
    ms = 1e3 * (time.perf_counter() - t0) / max(1, args.steps)
    sample = f"{nprop} proposal(s) x {N_PTS} pts per step (of the {B_PER_GPU}-proposal batch), fp32, torch CPU, {threads} threads"
    line = dict(metric=METRIC, value=val, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=ms,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=WORKLOAD, proposals_per_step=nprop, scene_points=N_PTS, template_points=N_PTS,
                            note="reference algorithm restated on the host (oracle port; the Python reference cannot travel)"),
                cpu_baseline=dict(value=val, unit=UNIT, cores=threads, kind="port", sample=sample),
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def run_scene(args):
    """BASELINE configs #4 / #5 -- STRONG scaling of one fixed piece of work over the ranks (SURVEY.md 8e):
      --workload ycbv  (config #5): one frame, 200 proposals, 21 objects x 42 templates x 1024-d descriptors.  Template scoring
                        is object-sharded (every rank scores all proposals against its objects with the fused CUDA kernel, one
                        12-byte-per-proposal all-gather picks the winners), PEM matching is proposal-sharded (200 / N per rank,
                        each proposal against the template bank of ITS object), one ragged all-gather of the poses.
      --workload lmo   (config #4): 8 scenes x 16 proposals, 8 objects: scenes are sharded over the ranks; per scene the SAM ViT-H
                        encoder (1024 x 1024), template scoring, PEM matching of its proposals; one all-gather of the poses.
    value = poses of the whole job / max-over-ranks time."""
    import torch.distributed as dist
    from sam6d_b200 import _lib, dist as sdist, ism, synth
    from sam6d_b200.pem import Net
    world, rank, local_rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ycbv = args.workload == "ycbv"
    O, T, C = (21, 42, 1024) if ycbv else (8, 42, 1024)
    scenes, P = (1, 200) if ycbv else (8, 16)
    net = Net(precision=args.precision).to(dev).eval()
    net.load_state_dict(synth.make_pem_state_dict(seed=1), strict=True)
    if not args.no_graph:
        net.enable_graphs()          # the per-rank chunk keeps its shape and (through the caching allocator) its buffers: replayed
    # template banks of the O objects (dense_po / dense_fo, 2048 points each) and per-scene proposals
    bank = synth.make_pem_inputs(B=O, n=N_PTS, n_model=N_MODEL, seed=50)
    bank_po, bank_fo, bank_model = bank["dense_po"].to(dev), bank["dense_fo"].to(dev), bank["model"].to(dev)
    sc = []
    for s_ in range(scenes):
        inp = synth.make_pem_inputs(B=P, n=N_PTS, n_model=N_MODEL, seed=200 + s_)
        q, r = synth.make_descriptors(P=P, O=O, T=T, C=C, seed=300 + s_)
        sc.append(dict(pts=inp["pts"].to(dev), dense_fm=inp["dense_fm"].to(dev), q=q.to(dev)))
    _, refs = synth.make_descriptors(P=4, O=O, T=T, C=C, seed=300)
    refs = refs.to(dev)
    o_lo, o_hi = sdist.shard_range(O, rank, world)
    refs_local = refs[o_lo:o_hi].contiguous()
    enc, frames = None, None
    if not ycbv:
        from sam6d_b200.sam import build_image_encoder
        enc = build_image_encoder("vit_h", precision=args.precision).to(dev).eval()
        g = torch.Generator().manual_seed(1)
        with torch.no_grad():
            for prm in enc.parameters():
                prm.copy_(torch.randn(prm.shape, generator=g) * (0.02 if prm.dim() > 1 else 0.05))
        frames = [synth.make_images(B=1, seed=400 + s_).to(dev) for s_ in range(scenes)]
    gen = torch.Generator(device=dev).manual_seed(1 + rank)

    def pem_on(scene, idx, obj):
        """proposals idx of a scene, each against the bank of its assigned object"""
        if idx.numel() == 0:
            return torch.zeros(0, sdist.POSE_FLOATS, device=dev)
        ep = dict(pts=scene["pts"][idx].contiguous(), dense_fm=scene["dense_fm"][idx].contiguous(), dense_po=bank_po[obj].contiguous(),
                  dense_fo=bank_fo[obj].contiguous(), model=bank_model[obj].contiguous())
        rand = torch.rand(idx.numel(), synth.N_PROPOSAL1 * 3, device=dev, generator=gen)
        return sdist.pack_poses(net(ep, rand=rand))

    def step(i):
        if ycbv:
            scene = sc[0]
            # every proposal keeps its best object (threshold -1: the sweep times all 200 poses, as BASELINE config #5 states)
            sel, obj, score, tmpl = sdist.sharded_semantic_score(scene["q"], refs_local, o_lo, confidence_thresh=-1.0)
            lo, hi = sdist.shard_range(P, rank, world)
            counts = [b - a for a, b in (sdist.shard_range(P, r_, world) for r_ in range(world))]
            local = pem_on(scene, sel[lo:hi], obj[lo:hi])
            return sdist.all_gather_poses(local, counts=counts)
        mine = list(range(rank, scenes, world))
        outs = []
        for s_ in mine:
            enc(frames[s_])
            sel, obj, score, tmpl = ism.compute_semantic_score(sc[s_]["q"], refs, confidence_thresh=-1.0)
            outs.append(pem_on(sc[s_], sel, obj))
        local = torch.cat(outs, dim=0) if outs else torch.zeros(0, sdist.POSE_FLOATS, device=dev)
        counts = [len(range(r_, scenes, world)) * P for r_ in range(world)]
        return sdist.all_gather_poses(local, counts=counts)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(i)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = step(i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    if rank == 0:
        total = scenes * P
        assert out.shape[0] == total
        line = dict(metric=METRIC, value=total * args.steps / (ms * 1e-3), unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype="bf16" if args.precision == "bf16" else "f32", data="synthetic",
                    config=dict(workload="ycbv_21obj_200proposals_template_parallel" if ycbv else "lmo_8scenes_x16proposals_ism_plus_pem",
                                objects=O, templates=T, proposals_per_step=total, scenes_per_step=scenes,
                                parallelism=(f"objects sharded x{world} for scoring (1 all-gather, 12 B/proposal/rank) + proposals sharded x{world} "
                                             f"for matching ({total // world}-{-(-total // world)} per GPU) + 1 ragged all-gather of poses") if ycbv else
                                            f"scenes sharded x{world} (SAM ViT-H encoder + scoring + matching per scene) + 1 all-gather of poses",
                                cache="per-step working set exceeds L2"),
                    gpu_launches=launches, clocks=sampler.summary() if sampler else None)
        if net._graphs is not None:
            line["config"]["launch"] = f"matching step replayed as a CUDA graph where the buffers recur ({net._graphs.captures} captures, {net._graphs.replays} replays on rank 0)"
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_ism(args):
    """BASELINE.json config #3: SAM ViT-H image encoder + 42-template cosine scoring on a batch of synthetic frames.
    Secondary line (the headline metric of the repo is the PEM poses/s line): python bench.py --workload ism"""
    from sam6d_b200 import _lib, ism, synth
    from sam6d_b200.sam import build_image_encoder
    assert torch.cuda.is_available()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    F_, P, O, T = args.batch if args.batch != B_PER_GPU else 16, 64, 8, 42
    enc = build_image_encoder("vit_h", precision=args.precision).to(dev).eval()
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for prm in enc.parameters():                           # seeded random weights of the ViT-H architecture
            prm.copy_(torch.randn(prm.shape, generator=g) * (0.02 if prm.dim() > 1 else 0.05))
        for m in enc.modules():
            if isinstance(m, torch.nn.LayerNorm) or m.__class__.__name__ == "LayerNorm2d":
                m.weight.fill_(1.0); m.bias.zero_()
    host = [synth.make_images(B=F_, seed=10 + s).pin_memory() for s in range(2)]
    resident = [h.to(dev) for h in host]
    q, r = synth.make_descriptors(P=F_ * P, O=O, T=T, C=1024, seed=3)
    qd, rd = q.to(dev), r.to(dev)
    qh = q.pin_memory()

    def step(i, e2e=False):
        img = host[i % 2].to(dev, non_blocking=True) if e2e else resident[i % 2]
        emb = enc(img)
        sel = ism.compute_semantic_score(qh.to(dev, non_blocking=True) if e2e else qd, rd)
        if e2e:
            return emb[:, :, 0, 0].cpu(), sel[3].cpu()
        return emb, sel

    def timed(steps, e2e):
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(i, e2e)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), _lib.launch_count() - l0

    for i in range(max(args.warmup, 3)):
        step(i)
    ms, launches = timed(args.steps, False)
    ms_e2e, _ = timed(args.steps, True)
    pk = peaks()
    flops = 5.96e12 * F_                                          # SURVEY.md 8d: 5.96 TFLOP per 1024^2 frame
    ach = flops * args.steps / (ms * 1e-3) / 1e12
    line = dict(metric="frames/sec", value=F_ * args.steps / (ms * 1e-3), unit="frames/s", n_gpus=1, steps=args.steps,
                warmup=max(args.warmup, 3), ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="bf16" if args.precision == "bf16" else "f32", data="synthetic",
                config=dict(workload="ism_sam_vith_encoder_plus_template_scoring", frames_per_step=F_, image="1024x1024 (640x480 frame resized+padded)",
                            proposals_per_frame=P, objects=O, templates=T, cache="activations per step (>3 GB) exceed L2"),
                e2e=dict(value=F_ * args.steps / (ms_e2e * 1e-3), unit="frames/s", h2d_bytes_per_step=host[0].numel() * 4 + qh.numel() * 4,
                         d2h_bytes_per_step=F_ * 256 * 4 + F_ * P * 8),
                gpu_launches=launches,
                roofline=dict(kernel="whole encoder (tcgen05 GEMMs + attention)", bound="tensor", achieved=ach, peak=pk["tensor"], unit="TFLOP/s",
                              frac=ach / pk["tensor"], traffic=None, peak_source=pk["source"] + " bf16_tflops_sustained"))
    if not args.no_cpu_baseline:
        from oracle import sam_oracle as so                # CPU leg only: the oracle port is the thing timed here
        threads = host_threads()
        torch.set_num_threads(threads)
        sd = {k: v.detach().cpu() for k, v in enc.state_dict().items()}
        t0 = time.perf_counter()
        with torch.no_grad():
            so.image_encoder(sd, host[0][:1].clone(), 16, (7, 15, 23, 31))
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = dict(value=1.0 / dt, unit="frames/s", cores=threads, kind="port",
                                    sample=f"1 of the {F_} frames through the full 32-block ViT-H encoder, one pass, {dt:.1f} s, torch fp32")
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the same-box reference lines (oracle port + reference _ext kernels on this GPU)")
    ap.add_argument("--batch", type=int, default=B_PER_GPU)
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every kernel of a step one by one instead of replaying the captured step (Net.enable_graphs)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="bf16: tcgen05 tensor-core kernels (bf16 operands, fp32 accumulate); fp32: CUDA-core exact path")
    ap.add_argument("--rgb", action="store_true",
                    help="PEM workload including the RGB branch (SURVEY 8f row N1): ViT-B/16 features of 224x224 crops + pixel "
                         "gather replace the given dense_fm; not the BASELINE configuration, reported as its own workload name")
    ap.add_argument("--workload", default="pem", choices=["pem", "ism", "ycbv", "lmo"],
                    help="pem: BASELINE config #2 (headline); ism: config #3, SAM ViT-H encoder + template scoring; ycbv / lmo: "
                         "configs #5 / #4, strong scaling of one fixed frame set over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the poses Net.forward returned in the last one (rank 0: init_R, init_t, "
                         "pred_R, pred_t, pred_pose_score) as DIR/<name>.npy, float32; the inputs are seeded, so two builds "
                         "compare output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "pem"):
        ap.error("--dump-outputs writes the outputs of the pem workload of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "ism":
        return run_ism(args)
    if args.workload in ("ycbv", "lmo"):
        return run_scene(args)

    import torch.distributed as dist
    from sam6d_b200 import synth                  # seeded weights + synthetic inputs (no oracle code on this arm)
    from sam6d_b200 import _lib, dist as sdist
    from sam6d_b200.graph import OUT_KEYS
    from sam6d_b200.pem import Net

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU: sam6d_b200 has no CPU fallback"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    B = args.batch

    if args.rgb:
        from sam6d_b200.vit import ViTEncoder
        enc = ViTEncoder(npoint=N_PTS, precision=args.precision)
        enc.load_state_dict(synth.make_vit_state_dict(seed=1), strict=True)
        net = Net(feature_extraction=enc, precision=args.precision).to(dev).eval()
        net.load_state_dict({**synth.make_pem_state_dict(seed=1), **{"feature_extraction." + k: v for k, v in enc.state_dict().items()}},
                            strict=True)
        keys = ("pts", "dense_po", "dense_fo", "model")
    else:
        net = Net(precision=args.precision).to(dev).eval()
        net.load_state_dict(synth.make_pem_state_dict(seed=1), strict=True)
        keys = ("pts", "dense_fm", "dense_po", "dense_fo", "model")
    host = [{k: v.pin_memory() for k, v in synth.make_pem_inputs(B=B, n=N_PTS, n_model=N_MODEL, seed=100 + rank * 7 + s).items()
             if k in keys} for s in range(2)]
    if args.rgb:
        g_rgb = torch.Generator().manual_seed(5 + rank)
        for h in host:
            h["rgb"] = torch.randn(B, 3, 224, 224, generator=g_rgb).pin_memory()
            h["rgb_choose"] = torch.randint(0, 224 * 224, (B, N_PTS), generator=g_rgb).pin_memory()
    graphs = not args.no_graph and not os.environ.get("SAM6D_PROFILE_ONE_STEP")
    if graphs:
        # repeated calls on the same input buffers replay one captured CUDA graph per input set (sam6d_b200/graph.py); the first
        # call on a buffer set runs launch by launch, the second captures -- both happen during warm-up
        net.enable_graphs()
    resident = [{k: v.to(dev) for k, v in h.items()} for h in host]
    h2d_bytes = sum(v.numel() * v.element_size() for v in host[0].values())
    gen = torch.Generator(device=dev).manual_seed(1 + rank)

    last = {}

    def step_resident(i):
        ep = dict(resident[i % 2])
        rand = torch.rand(B, synth.N_PROPOSAL1 * 3, device=dev, generator=gen)
        out = net(ep, rand=rand)
        last["out"] = out
        poses = sdist.pack_poses(out)
        return sdist.all_gather_poses(poses)

    host_out = torch.empty(world * B, sdist.POSE_FLOATS).pin_memory()

    # end to end through the public API (Net.forward on a dict of device tensors): every step copies its inputs from pinned
    # host memory and reads its poses back.  The copies run on a second stream into the other half of a double buffer, so
    # step i+1's inputs arrive while step i computes (K host->device copies and K read-backs inside the timed region).
    copy_stream = torch.cuda.Stream(dev)
    dev_in = [{k: torch.empty_like(v, device=dev) for k, v in h.items()} for h in host]
    copied, computed, pipe = [None, None], [None, None], {"next": 0}

    def issue_copy(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            if computed[s] is not None:
                copy_stream.wait_event(computed[s])          # the step that last read this buffer has finished
            for k, v in host[s].items():
                dev_in[s][k].copy_(v, non_blocking=True)
            copied[s] = torch.cuda.Event()
            copied[s].record(copy_stream)
        pipe["next"] = i + 1

    def step_e2e(i):
        if pipe["next"] <= i:
            issue_copy(i)
        torch.cuda.current_stream().wait_event(copied[i % 2])
        if i + 1 < args.steps:
            issue_copy(i + 1)
        rand = torch.rand(B, synth.N_PROPOSAL1 * 3, device=dev, generator=gen)
        out = net(dict(dev_in[i % 2]), rand=rand)
        poses = sdist.all_gather_poses(sdist.pack_poses(out))
        host_out.copy_(poses, non_blocking=True)
        computed[i % 2] = torch.cuda.Event()
        computed[i % 2].record()
        return poses

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile_kernel=None):
        barrier()
        names = [profile_kernel] if isinstance(profile_kernel, str) else list(profile_kernel or [])
        for nm in names:
            _lib.time_kernel(nm, True)
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - l0
        kernel_ms = None
        if names:
            kernel_ms = {}
            for nm in names:
                kernel_ms[nm] = [a.elapsed_time(b) for a, b in _lib.timed_events(nm)]
                _lib.time_kernel(nm, False)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, launches, kernel_ms

    n_warm = max(args.warmup, 3)
    n_warm_run = max(n_warm, 4) if graphs else n_warm          # two input sets: sighting, capture (+ first replay) of each
    for i in range(n_warm_run):
        step_resident(i)
    if os.environ.get("SAM6D_PROFILE_ONE_STEP"):
        # ncu --profile-from-start off: capture exactly one warmed-up step
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident(0)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, _ = timed(step_resident, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: last["out"][k] for k, _ in OUT_KEYS})
    # dominant-kernel roofline: same steps again with CUDA events around every launch of the kernels the roofline report names
    # (the stream over E; the attention kernel that consumes its scores; the geometric-embedding kernel that writes E)
    from sam6d_b200 import pem as _pem
    rpe_name = "sam6d_rpe_scores_tc" if (args.precision == "bf16" and _pem.RPE_TC) else "sam6d_rpe_scores"
    padded = rpe_name == "sam6d_rpe_scores_tc" and _pem.PADDED_BIAS
    if padded:
        rpe_name = "sam6d_rpe_scores_tc_ld"              # score planes with padded rows, consumed by sam6d_attn_tc_bias_ld
    # (launch by launch: the events bracket single launches, which a graph replay does not expose; same kernels, same inputs)
    step_graphs, net._graphs = net._graphs, None
    _, _, kall = timed(step_resident, args.steps,
                       profile_kernel=[rpe_name, "sam6d_attn_tc", "sam6d_attn_tc_bias_ld", "sam6d_geo_embed_tc", "sam6d_geo_embed_lut"])
    net._graphs = step_graphs
    kms = kall[rpe_name]
    for i in range(4 if graphs else 2):
        step_e2e(i)
    torch.cuda.synchronize()
    pipe["next"], computed[0], computed[1] = 0, None, None     # the timed run issues all of its own copies
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)

    if rank == 0:
        pk = peaks()
        S = net.coarse_npoint + 1
        e_size = 2 if args.precision == "bf16" else 4
        # 12 RPE self-attention calls per forward (SURVEY 8a4); the scene and template clouds share one launch when they are
        # batched, so a launch streams the embedding of `clouds` point clouds exactly once
        clouds = B * 12 * args.steps // len(kms)
        e_bytes = clouds * S * S * 256 * e_size
        # SURVEY.md 8(d): algorithmic bytes of an RPE self-attention call = the pair embedding E read once + the token matrix
        # (636 MB + 3.2 MB per 32-cloud call in bf16).  The score tensor that rpe_scores hands to the attention kernel is NOT
        # algorithmic (it exists only because scores and softmax are two kernels) and is not counted.
        alg_bytes = e_bytes + clouds * S * 256 * e_size
        k_avg_ms = sum(kms) / len(kms)
        achieved = alg_bytes / (k_avg_ms * 1e-3) / 1e9
        # whole RPE attention = score stream + the tensor-core attention launch that adds them as a dense bias (every third
        # sam6d_attn_tc call of a block: self, cross, cross)
        att = kall.get("sam6d_attn_tc") or []
        att_bias = att[0::3] if len(att) == 3 * len(kms) else []
        if padded:
            att_bias = kall.get("sam6d_attn_tc_bias_ld") or []
        att_avg_ms = sum(att_bias) / len(att_bias) if att_bias else None
        attention_frac = alg_bytes / ((k_avg_ms + att_avg_ms) * 1e-3) / 1e9 / pk["hbm"] if att_avg_ms else None
        geo = kall.get("sam6d_geo_embed_tc") or []
        roofline_tensor = None
        if geo:
            geo_ms = sum(geo) / len(geo)                 # one call per step = both launches (distance pass + angle pass)
            # SURVEY.md 8(d) "min" count: proj_a on the 3 angle rows of every pair, 2*B clouds (the distance projection can be folded)
            flops_min = 2.0 * (2 * B) * S * S * 3 * 256 * 256
            flops_issued = 2.0 * (2 * B) * S * S * 5 * 256 * 256          # 4 angle rows (1 padding) + 1 distance row per pair
            roofline_tensor = dict(kernel="geo_embed_tc_kernel<1> + <0> (GeometricStructureEmbedding: writes E)", bound="tensor",
                                   achieved=flops_min / (geo_ms * 1e-3) / 1e12, peak=pk["tensor"], unit="TFLOP/s",
                                   frac=flops_min / (geo_ms * 1e-3) / 1e12 / pk["tensor"], avg_call_ms=geo_ms,
                                   flops_min_per_call=flops_min, flops_issued_per_call=flops_issued,
                                   share_of_step=sum(geo) / ms)
        roofline_geo = None
        lut = kall.get("sam6d_geo_embed_lut") or []
        if lut:
            # table-interpolation kernel (csrc/geo_lut.cu): no MMA left, E is written exactly once -> HBM-write bound.  Algorithmic
            # bytes = E (2B clouds x S x S x 256 bf16) + the four fp32 indices per pair it reads
            lut_ms = sum(lut) / len(lut)
            geo_bytes = (2 * B) * S * S * (256 * 2 + 16)
            roofline_geo = dict(kernel="geo_embed_lut_kernel (GeometricStructureEmbedding by table interpolation: writes E once)", bound="hbm",
                                achieved=geo_bytes / (lut_ms * 1e-3) / 1e9, peak=pk["hbm"], unit="GB/s",
                                frac=geo_bytes / (lut_ms * 1e-3) / 1e9 / pk["hbm"], avg_launch_ms=lut_ms,
                                algorithmic_bytes_per_launch=geo_bytes, share_of_step=sum(lut) / ms,
                                note="replaces the tcgen05 projections (977 GFLOP min per step, 1.30 ms = 0.53 of the sustained bf16 rate): "
                                     "the projected embedding of one scalar is tabulated, so the flops are gone rather than run faster")
        value = world * B * args.steps / (ms * 1e-3)
        e2e_val = world * B * args.steps / (ms_e2e * 1e-3)
        traffic = None
        prof = os.path.join(ROOT, "profiles", "rpe_scores_traffic.json")
        if os.path.exists(prof):
            rec = json.load(open(prof)).get("bf16" if args.precision == "bf16" else "fp32", {})
            traffic = rec.get("dram_bytes_per_launch")
            if traffic is not None and rec.get("clouds_per_launch", B) != clouds:      # ncu capture of another launch shape
                traffic = None
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=n_warm, warmup_run=n_warm_run,
            ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="bf16" if args.precision == "bf16" else "f32", data="synthetic",
            config=dict(workload=WORKLOAD + ("+vitb_rgb_branch" if args.rgb else ""), proposals_per_gpu=B, scene_points=N_PTS, template_points=N_PTS, sparse_points=net.coarse_npoint,
                        feat_dim=C_FEAT, model_points=N_MODEL, parallelism=f"proposal-sharded x{world}, 1 all-gather of poses",
                        cache="inputs+intermediates per step (>1 GB) exceed the 126 MB L2; two input sets alternate",
                        launch=(f"one CUDA-graph replay per step ({launches // args.steps} kernels each, captured from Net.forward; "
                                f"{step_graphs.captures} graphs, {step_graphs.replays} replays in this run)") if graphs and step_graphs
                        else "kernel by kernel"),
            e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=h2d_bytes, d2h_bytes_per_step=world * B * sdist.POSE_FLOATS * 4,
                     ms_per_step=ms_e2e / args.steps),
            gpu_launches=launches,
            roofline=dict(kernel=f"{rpe_name[6:]} ({'bf16' if args.precision == 'bf16' else 'fp32'} E; PEM RPE attention, streams the geometric embedding)", bound="hbm",
                          achieved=achieved, peak=pk["hbm"], unit="GB/s", frac=achieved / pk["hbm"], traffic=traffic,
                          peak_source=pk["source"] + " (MEASURED_PEAKS.json hbm_gbs)" if pk["source"] == "measured" else "fallback 6650 GB/s",
                          algorithmic_bytes_per_launch=alg_bytes, clouds_per_launch=clouds, launches_timed=len(kms), avg_launch_ms=k_avg_ms,
                          share_of_step=sum(kms) / ms,
                          attention_frac=attention_frac, attention_avg_ms=(k_avg_ms + att_avg_ms) if att_avg_ms else None,
                          attention_note="score stream + the attn_tc launch that consumes it (softmax, PV), same algorithmic bytes"),
            roofline_tensor=roofline_tensor,
            roofline_geo=roofline_geo,
            clocks=sampler.summary() if sampler else None,
        )
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            cpu_oracle_throughput(1, threads, 1)
            val, times = cpu_oracle_throughput(2, threads)
            line["cpu_baseline"] = dict(value=val, unit=UNIT, cores=threads, kind="port",
                                        sample=f"{CPU_SAMPLE_B} of the {B} proposals, 2 timed passes after a 1-proposal warm-up, "
                                               f"{sum(times):.1f} s of CPU work, torch fp32 on {threads} threads")
        if world == 1 and not args.no_ref_gpu:
            line["same_box_reference"] = same_box_reference(dev, B)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
