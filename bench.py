#!/usr/bin/env python
"""bench.py -- latent-volume denoise steps/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host CPU (oracle port)
  python bench.py ... --dump-outputs DIR                   # + the latents of the last timed step, DIR/*.npy (float32)

Workload (BASELINE.json configs[1], SURVEY cfg-2): conditional_dm3d U-Net (F=32, widths 64/128/256, cross-attention at
8^3), DDPM, batch 8 per GPU, 32^3 x 256 latent, class-id context, random-init weights, synthetic latents.
A "step" = one reverse-diffusion step of the whole batch (U-Net forward + fused posterior update);
value = volumes * steps / second over all GPUs (weak scaling: independent sample batches per GPU, no collective).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "latent-volume denoise steps/sec"
UNIT = "volume-steps/s"
CFG = dict(S=32, C_lat=256, B=8, T=1000)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return dict(hbm=j["hbm_gbs"], tf=j["bf16_tflops"], tf_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
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
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
        return dict(sm_mhz=float(np.median(busy)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)),
                    samples=len(sm), reasons=sorted(reasons))


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo", rank=rank, world_size=world)
    return world, rank, local


def max_over_ranks(v, world, device):
    if world == 1:
        return v
    import torch.distributed as dist
    t = torch.tensor([v], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


# ----------------------------------------------------------------------------------------------- CPU (reference) arm
def oracle_cpu_rate(steps, warmup, budget_s=90.0, batch=None):
    """The reference's algorithm for this path on the host CPU (oracle port: PyTorch-CPU fp32 restatement of
    conditional_dm3d.build_model + DiffusionModel.sample; TensorFlow is not installable here).  Bounded sample:
    a few DDPM steps of the cfg-2 workload at ``batch`` volumes per step (default: the workload's own 8), all host threads."""
    Bc = batch or CFG["B"]
    from oracle.unet import UNet as OUNet
    from oracle import init as OI, sampler as OS
    from oracle.schedule import Betas
    torch.set_num_threads(os.cpu_count() or 1)
    S, C = CFG["S"], CFG["C_lat"]
    ou = OUNet(S, C, [64, 128, 256], [False, False, True, True], first_conv_channels=32, conditional=True)
    P = OI.make_params(ou.spec(), 0, "keras")
    b = Betas(CFG["T"])
    x = OI.normal((Bc, S, S, S, C), 1)
    ctx = torch.arange(Bc) % 2
    z = OI.normal((Bc, S, S, S, C), 2)

    def one(t):
        nonlocal x
        with torch.no_grad():
            eps = ou.forward(P, x, torch.full((Bc,), t), ctx=ctx)
            x = OS.ddpm_step(b, x, eps, t, z)

    t0 = time.perf_counter()
    one(CFG["T"] - 1)
    first = time.perf_counter() - t0
    w = max(0, min(warmup - 1, int(budget_s * 0.2 / max(first, 1e-3))))
    for i in range(w):
        one(CFG["T"] - 2 - i)
    n = max(1, min(steps, int(budget_s / max(first, 1e-3))))
    t0 = time.perf_counter()
    for i in range(n):
        one(CFG["T"] - 2 - w - i)
    dt = time.perf_counter() - t0
    return dict(rate=Bc * n / dt, steps=n, warmup=w + 1, ms_per_step=1e3 * dt / n, cores=torch.get_num_threads(), batch=Bc,
                sample=f"{Bc} volumes x {n} DDPM steps of cfg-2 (32^3x256 latent, conditional U-Net, per-sample class ids), PyTorch-CPU fp32 oracle port")


def run_reference(args):
    world, rank, local = dist_setup(args.gpus)
    if rank != 0:
        barrier(world)
        return
    r = oracle_cpu_rate(args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["rate"], "unit": UNIT, "n_gpus": args.gpus, "steps": r["steps"],
            "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(1, per_step_volumes=r["batch"]),
            "cpu_baseline": {"value": r["rate"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["rate"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference = TensorFlow/Keras (not installable offline): timed its CPU restatement (oracle/) on the host cores; rank 0 only"}
    print(json.dumps(line), flush=True)
    barrier(world)


def workload_config(n_gpus, per_step_volumes=None):
    return {"workload": "cfg-2: conditional_dm3d U-Net, DDPM T=1000, 32^3x256 latent, class-id context, batch 8 per GPU",
            "latent": [CFG["S"]] * 3 + [CFG["C_lat"]], "batch_per_gpu": CFG["B"] if per_step_volumes is None else per_step_volumes,
            "global_batch": (CFG["B"] if per_step_volumes is None else per_step_volumes) * n_gpus, "timesteps": CFG["T"],
            "parallelism": f"independent sample batches x{n_gpus} (no collective on the sampling path)",
            "l2": "not flushed: one step touches >10 GB of activations+weights, far larger than the 126 MB L2"}


# ----------------------------------------------------------------------------------------------- CUDA arm
def ncu_traffic():
    """Per-launch DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel family from the committed
    ncu --set full capture of this same command (profiles/r2_traffic.json, written by tools/ncu_traffic.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            return json.load(f)
    except OSError:
        return None


DUMP_ELEMS = 1 << 23   # 32 MB of fp32 per rank


def dump_outputs(out_dir, lat, rank, world):
    """Write the fp32 latents the timed steps left in the step state (what generate() returns to its caller) to
    <out_dir>/latents.npy, or, when larger than DUMP_ELEMS, DUMP_ELEMS of them at flat indices drawn once from a seed-0 CPU
    generator and sorted (latents_sample.npy), so that two builds can be compared output for output."""
    flat = lat.reshape(-1)
    name = "latents"
    if flat.numel() > DUMP_ELEMS:
        idx = torch.randint(0, flat.numel(), (DUMP_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
        flat, name = flat[idx.to(flat.device)], "latents_sample"
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + (f"_rank{rank}" if world > 1 else "") + ".npy"), flat.float().cpu().numpy())


def event_time(fn, iters, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def run_ours(args):
    world, rank, local = dist_setup(args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import b200dm
    from b200dm import _lib as L, ops

    S, C, B, T = CFG["S"], CFG["C_lat"], CFG["B"], CFG["T"]
    K, W = args.steps, max(args.warmup, 3)
    a = types.SimpleNamespace(timesteps=T, num_gpus=world, kernel_resize=False, bs=B * world)
    # first stage of the sampling + decode job (north_star; BASELINE configs[2]): vqgan_attn_cp quantizer (K=1024, D=256) + Decoder
    # (32,64,128): 32^3 x 256 latents -> 128^3 x 1 volumes
    fs = b200dm.VQGAN(num_channels=(32, 64, 128), num_embeddings=1024, embedding_dim=C)
    dm = b200dm.ConditionalDiffusionModel(S, 1024, C, None, a, first_stage=fs)
    shape = (B, S, S, S, C)
    sid0 = rank * B
    ctx = (torch.arange(B) + sid0) % 2
    # ---- public-API warm-up: compiles the program, captures the step graph, runs W+ steps
    lat = dm.generate(shape, last_step=T - W, seed=1234, sample_id0=sid0, context=ctx)
    assert torch.isfinite(lat).all(), "non-finite latents"
    assert L.debug_flag() == 0, "tcgen05/TMA watchdog fired"
    st = dm._step
    graph, nets = st["graph"], st["nets"]
    # per chain: U-Net program (+ the update kernel unless it is fused into the output conv's epilogue); + t advance
    launches_per_step = sum(net.prog.num_launches + (0 if st["fused"] else 1) for net in nets) + 1

    def reset(t0=T - 1):   # restart the device-side timestep walker on the DDPM sequence T-1, T-2, ...
        st["t_seq"].copy_(torch.tensor(list(range(T - 1, -1, -1)) + [-1, -1], dtype=torch.int32))
        st["t_dev"][:4].copy_(torch.tensor([t0, t0 - 1, T - 1 - t0, 0], dtype=torch.int32))

    # ---- device-resident timing: K graph replays between CUDA events on the launching stream
    reset()
    for _ in range(W):
        graph.replay()
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.3)
    barrier(world)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
    clk = clocks.stop()
    value = world * B * K / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, st["x"], rank, world)

    # ---- end to end through the public API with HOST buffers: pinned x_T -> H2D -> K steps -> D2H latents
    x_host = torch.randn(shape, generator=torch.Generator().manual_seed(rank)).pin_memory()
    out_host = torch.empty(shape, dtype=torch.float32).pin_memory()
    dm.generate(shape, last_step=T - 2, x_T=x_host, seed=1234, sample_id0=sid0, context=ctx)  # warm the path
    barrier(world)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lat = dm.generate(shape, last_step=T - K, x_T=x_host, seed=1234, sample_id0=sid0, context=ctx)
    out_host.copy_(lat, non_blocking=True)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, world, dev)
    barrier(world)
    nbytes = x_host.numel() * 4
    e2e = {"value": world * B * K / e2e_s, "unit": UNIT, "h2d_bytes_per_step": nbytes / K, "d2h_bytes_per_step": nbytes / K,
           "call": "ConditionalDiffusionModel.generate(shape, last_step=T-K, x_T=<pinned host>, context=ids) -> host latents"}

    # ---- the sampling + decode job (north_star's scaling target), through the public API with host buffers:
    #      generate(K steps) -> quantize -> vqgan_attn_cp decoder -> host volumes
    vol_host = torch.empty(B, 128, 128, 128, 1, dtype=torch.float32).pin_memory()

    def sample_decode(last_step):
        lat_ = dm.generate(shape, last_step=last_step, x_T=x_host, seed=1234, sample_id0=sid0, context=ctx)
        vol_host.copy_(dm.decode(lat_, quantize=True), non_blocking=True)
        torch.cuda.synchronize()

    sample_decode(T - 2)   # compiles the decoder program
    assert torch.isfinite(vol_host).all() and L.debug_flag() == 0
    barrier(world)
    t0 = time.perf_counter()
    sample_decode(T - K)
    sd_s = max_over_ranks(time.perf_counter() - t0, world, dev)
    barrier(world)
    e2e_sd = {"value": world * B * K / sd_s, "unit": UNIT, "volumes_per_s": world * B / sd_s, "seconds": sd_s, "steps": K,
              "h2d_bytes": nbytes, "d2h_bytes": vol_host.numel() * 4,
              "call": "generate(last_step=T-K, x_T=<pinned host>) -> decode(latents, quantize=True) [VQ K=1024 + vqgan_attn_cp decoder 32^3->128^3] -> host volumes"}

    # ---- sustained: the FULL 1000-step chain (device-resident replay, ~3 s) with its own clock record, and the whole
    #      1000-step sampling + decode job through the public API
    sustained = None
    if not args.no_sustained:
        reset()
        c2 = ClockSampler(local)
        c2.start()
        time.sleep(0.2)
        barrier(world)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(T):
            graph.replay()
        s1.record()
        torch.cuda.synchronize()
        barrier(world)
        s_ms = max_over_ranks(s0.elapsed_time(s1), world, dev)
        c2r = c2.stop()
        barrier(world)
        t0 = time.perf_counter()
        sample_decode(0)
        job_s = max_over_ranks(time.perf_counter() - t0, world, dev)
        barrier(world)
        sustained = {"steps": T, "ms_per_step": s_ms / T, "value": world * B * T / (s_ms * 1e-3), "unit": UNIT, "clocks": c2r,
                     "job_1000_steps_plus_decode": {"seconds": job_s, "volumes_per_s": world * B / job_s,
                                                    "volume_steps_per_s": world * B * T / job_s, "volumes": world * B,
                                                    "call": "generate(shape, x_T=<pinned host>) [T=1000] -> decode(quantize=True) -> host volumes"}}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": L.precision(), "data": "synthetic",
            "config": dict(workload_config(world), chains=st["chains"], storage=L.precision()), "clocks": clk, "e2e": e2e,
            "e2e_sample_decode": e2e_sd, "gpu_launches": launches_per_step * K}
    if sustained:
        line["sustained"] = sustained

    if rank == 0:
        # ---- roofline of the dominant kernel family: per-launch CUDA events over one more step
        pk = peaks()
        # burst conditions (SM clock at its maximum, no power cap) -> the burst cuBLAS figure is the honest denominator; the
        # sustained one (taken at ~1290 MHz under the power cap) only when the sampler saw the clock drop
        at_max = clk.get("sm_mhz") and clk.get("sm_max_mhz") and clk["sm_mhz"] >= 0.97 * clk["sm_max_mhz"]
        tf_peak, tf_src = (pk["tf"], "bf16_tflops (burst: SM clock at max during the timed region)") if at_max else \
            (pk["tf_sustained"], "bf16_tflops_sustained (SM clock below max during the timed region)")
        reset()
        rows = []
        for net in nets:          # every chain's program, one launch at a time with an event pair around each
            net.prog.run_timed()
            rows += net.prog.run_timed()
        tot_ms = sum(r[3] for r in rows)

        def agg(kinds):
            sel = [r for r in rows if r[0] in kinds]
            ms_, work = sum(r[3] for r in sel), sum(r[2] for r in sel)
            return sel, ms_, work

        sel, h_ms, h_fl = agg(("conv_halo",))
        ach = h_fl / (h_ms * 1e-3) / 1e12
        # (out.conv carries the whole posterior update in its epilogue when that is fused: it also gets a block of its own below)
        plain = [r for r in sel if not (st["fused"] and r[1] == "out.conv")]
        tr = ncu_traffic()
        x_elems = st["x"][:st["chain_batch"]].numel()
        # the fused out.conv reads x_t and writes x_{t-1} (fp32) + its 16-bit copy instead of writing eps: 4 + 4 + 2 bytes per element
        fused_bytes = x_elems * (4.0 + 4.0 + 2.0) + nets[0].prog.op_bytes.get("out.conv", 0.0) - x_elems * 4.0
        halo_alg_bytes = sum(fused_bytes if (st["fused"] and r[1] == "out.conv") else nets[0].prog.op_bytes.get(r[1], 0.0)
                             for r in sel) / max(1, len(sel))   # operands read once + outputs written once
        line["roofline"] = {"kernel": "conv_halo_kernel / conv_halo_up_kernel (persistent tcgen05 implicit-GEMM 3^3 Conv3D, TMA halo slabs): all launches of one step" +
                                      (" (out.conv included: its epilogue also runs the posterior update, see roofline_out_conv_fused_update)" if st["fused"] else ""),
                            "frac_without_fused_out_conv": sum(r[2] for r in plain) / (sum(r[3] for r in plain) * 1e-3) / 1e12 / tf_peak,
                            "bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak,
                            "peak_source": f"{pk['src']} MEASURED_PEAKS.json {tf_src}", "frac_of_sustained_peak": ach / pk["tf_sustained"],
                            "frac_of_burst_peak": ach / pk["tf"],
                            "traffic": (tr or {}).get("halo_bytes_per_launch"), "traffic_source": (tr or {}).get("source"),
                            "algorithmic_bytes_per_launch": halo_alg_bytes,
                            "launches": len(sel), "avg_launch_ms": h_ms / max(1, len(sel)),
                            "algorithmic_gflop_per_launch_avg": h_fl / 1e9 / max(1, len(sel)), "share_of_step": h_ms / tot_ms,
                            "timing": "CUDA events around every launch on the launching stream (b200dm_program_run_timed)"}
        sel, t_ms, t_fl = agg(("conv_halo", "conv", "attn"))
        line["roofline_all_tensor_kernels"] = {"kernels": "conv_halo(_up)_kernel + conv_igemm_kernel (1^3 / strided / parity convs, GEMMs) + flash_attn_kernel",
                                               "bound": "tensor", "achieved": t_fl / (t_ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                                               "frac": t_fl / (t_ms * 1e-3) / 1e12 / tf_peak, "launches": len(sel),
                                               "algorithmic_gflop_per_step": t_fl / 1e9, "share_of_step": t_ms / tot_ms}
        line["roofline_step"] = {"bound": "tensor", "achieved": t_fl / (ms / K * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                                 "frac": t_fl / (ms / K * 1e-3) / 1e12 / tf_peak,
                                 "note": "all algorithmic conv/attention FLOPs of one step / the graph-replayed step time (everything included)"}
        sel, e_ms, e_by = agg(("norm_act", "layernorm", "gn_stats", "softmax"))
        if sel:
            line["roofline_hbm_kernels"] = {"kernels": "norm_act / layernorm (fused elementwise passes left in the step)", "bound": "hbm",
                                            "achieved": e_by / (e_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                            "frac": e_by / (e_ms * 1e-3) / 1e9 / pk["hbm"], "launches": len(sel), "share_of_step": e_ms / tot_ms}
        # the posterior update: on the graph path it runs inside out.conv's epilogue (no launch of its own); the stand-alone
        # kernel (injected-noise / eps-callback path) is timed alone on scratch buffers against SURVEY 8(d)'s algorithmic bytes
        net0 = nets[0]
        xs = st["x"][:st["chain_batch"]]
        if st["fused"]:
            oc = next(r for r in rows if r[1] == "out.conv")
            f_bytes = fused_bytes   # x_t, x_{t-1}, 16-bit copy + the conv's input and weights
            line["roofline_out_conv_fused_update"] = {
                "kernel": "conv_halo_kernel<128,2,..,CG2,FUSE_UPD> (out.conv 64->256 3^3 + DDPM posterior + in-register Philox noise in the epilogue)",
                "avg_launch_ms": oc[3], "tensor": {"achieved": oc[2] / (oc[3] * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s", "frac": oc[2] / (oc[3] * 1e-3) / 1e12 / tf_peak},
                "hbm": {"achieved": f_bytes / (oc[3] * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s", "frac": f_bytes / (oc[3] * 1e-3) / 1e9 / pk["hbm"],
                        "algorithmic_bytes_per_launch": f_bytes},
                "traffic": (ncu_traffic() or {}).get("fused_out_conv_bytes_per_launch"),
                "note": "replaces out.conv (fp32 eps out) + update_kernel (eps in): the fp32 eps round trip (2 x 4 B/element) never touches HBM"}
            xs = xs.clone()
            upd_eps, upd_xb = torch.zeros_like(xs), torch.empty_like(net0.x_in)
        else:
            upd_eps, upd_xb = st.get("update_eps", net0.eps), net0.x_in
        reset()

        def upd():
            L.check(L.lib().b200dm_ddpm_update(ctypes.byref(st["descs"][0]), L.ptr(xs), L.ptr(upd_eps), None, L.ptr(xs), L.ptr(upd_xb), L.stream()))

        u_ms = event_time(upd, 10, 3)
        u_alg = xs.numel() * (4.0 + 2.0 + 4.0 + 2.0)          # SURVEY 8(d): x_t fp32 + eps 16-bit + x_{t-1} fp32 + 16-bit copy
        u_moved = xs.numel() * (4.0 + upd_eps.element_size() + 4.0 + 2.0)
        line["roofline_update_kernel"] = {"kernel": "update_kernel (fused DDPM posterior + in-register Philox noise)" +
                                          (" -- stand-alone form; NOT in the timed step, where the update runs in out.conv's epilogue" if st["fused"] else ""),
                                          "bound": "hbm", "achieved": u_alg / (u_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                          "frac": u_alg / (u_ms * 1e-3) / 1e9 / pk["hbm"], "algorithmic_bytes_per_launch": u_alg,
                                          "bytes_moved_per_launch": u_moved, "moved_gbps": u_moved / (u_ms * 1e-3) / 1e9,
                                          "avg_launch_ms": u_ms, "working_set": "> 126 MB L2"}
        del upd_eps, upd_xb
        big = max((r for r in rows if r[0] == "norm_act"), key=lambda r: r[2], default=None)
        if big is not None:
            line["roofline_largest_norm_pass"] = {"kernel": f"norm_act_kernel ({big[1]})", "bound": "hbm", "achieved": big[2] / (big[3] * 1e-3) / 1e9,
                                                  "peak": pk["hbm"], "unit": "GB/s", "frac": big[2] / (big[3] * 1e-3) / 1e9 / pk["hbm"],
                                                  "algorithmic_bytes_per_launch": big[2], "avg_launch_ms": big[3]}
        if not args.no_cfg3:
            # secondary configurations: a failure here is reported in the line, it does not take the headline measurement with it
            for key, fn in (("cfg3", lambda: cfg3_line(b200dm, L, dev, pk, tf_peak)), ("cfg4", lambda: cfg4_line(b200dm, L, dev, tf_peak))):
                try:
                    line[key] = fn()
                except Exception as e:   # noqa: BLE001
                    line[key] = {"error": f"{type(e).__name__}: {e}"}
                    L.debug_flag()       # (read-and-reset)
                    torch.cuda.synchronize()
        if world == 1 and not args.no_cpu:
            r = oracle_cpu_rate(3, 1, budget_s=25.0)   # 8 volumes per step, like the GPU arm
            line["cpu_baseline"] = {"value": r["rate"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]}
        if args.dump_ops:
            with open(args.dump_ops, "w") as f:
                for r in rows:
                    f.write(f"{r[0]},{r[1]},{r[2]:.6g},{r[3]:.6f}\n")
        print(json.dumps(line), flush=True)
    barrier(world)


def cfg3_line(b200dm, L, dev, pk, tf_peak):
    """BASELINE configs[2]: VQ quantize (K=1024, D=256) + vqgan_attn_cp Decoder (32,64,128), 32^3 latents -> 128^3 volumes, batch 16,
    device-resident (CUDA events), with per-kernel rooflines from per-launch events."""
    Bd, s, D, Kc = 16, 32, 256, 1024
    vq = b200dm.VQGAN(num_channels=(32, 64, 128), num_embeddings=Kc, embedding_dim=D)
    z = torch.randn(Bd, s, s, s, D, device=dev) * 0.05
    q, idx, perp = vq.quantizer.quantize(z)
    vol = vq.decoder(q)
    flag = L.debug_flag()
    assert torch.isfinite(vol).all() and flag == 0 and tuple(vol.shape) == (Bd, 128, 128, 128, 1), f"cfg-3: watchdog flag {flag:#x}"
    ms_q = event_time(lambda: vq.quantizer.quantize(z), 3, 1)
    ms_d = event_time(lambda: vq.decoder.prog.run(), 5, 2)
    vq.decoder.prog.run_timed()
    rows = vq.decoder.prog.run_timed()
    N = Bd * s ** 3
    out = {"workload": "cfg-3: VQ quantize (K=1024, D=256) + vqgan_attn_cp Decoder (32,64,128): 32^3x256 -> 128^3x1, batch 16",
           "quantize_ms": ms_q, "decode_ms": ms_d, "volumes_per_s": Bd / ((ms_q + ms_d) * 1e-3), "decode_volumes_per_s": Bd / (ms_d * 1e-3),
           "vq_rows_per_s": N / (ms_q * 1e-3)}
    vq_fl, vq_by = 2.0 * N * Kc * D, N * D * 4.0 * 2 + N * 8.0 + Kc * D * 4.0
    out["roofline_vq"] = {"kernel": "vq_tc_kernel (tcgen05 fp16 hi/lo candidate search, 3 MMA passes = 3x the algorithmic FLOPs executed, + exact fp32 recheck + gather); indices bit-identical to the fp32 SIMT vq_kernel", "bound": "tensor", "achieved": vq_fl / (ms_q * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                          "frac": vq_fl / (ms_q * 1e-3) / 1e12 / tf_peak, "hbm_gbps": vq_by / (ms_q * 1e-3) / 1e9, "hbm_frac": vq_by / (ms_q * 1e-3) / 1e9 / pk["hbm"],
                          "note": "2*N*K*D FLOP vs the dense bf16 tensor peak and N*D*4*2 + N*8 + K*D*4 bytes vs HBM (SURVEY 8d: compute-bound at K=1024)"}
    tens = [r for r in rows if r[0] in ("conv", "conv_halo")]
    t_ms, t_fl = sum(r[3] for r in tens), sum(r[2] for r in tens)
    out["roofline_decoder_convs"] = {"bound": "tensor", "achieved": t_fl / (t_ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                                     "frac": t_fl / (t_ms * 1e-3) / 1e12 / tf_peak, "launches": len(tens), "ms": t_ms, "algorithmic_gflop": t_fl / 1e9}
    hb = [r for r in rows if r[0] in ("norm_act", "gn_stats", "stencil")]
    if hb:
        h_ms, h_by = sum(r[3] for r in hb), sum(r[2] for r in hb)
        out["roofline_decoder_hbm_passes"] = {"bound": "hbm", "achieved": h_by / (h_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                              "frac": h_by / (h_ms * 1e-3) / 1e9 / pk["hbm"], "launches": len(hb), "ms": h_ms}
    out["decoder_whole"] = {"algorithmic_gflop": t_fl / 1e9, "achieved_tflops": t_fl / (ms_d * 1e-3) / 1e12, "frac": t_fl / (ms_d * 1e-3) / 1e12 / tf_peak}
    out["top_ops"] = [{"kind": r[0], "op": r[1], "ms": round(r[3], 4)} for r in sorted(rows, key=lambda r: -r[3])[:8]]
    return out


def cfg4_line(b200dm, L, dev, tf_peak):
    """BASELINE configs[3]: dm3d U-Net with self-attention at the highest latent resolution (has_attention=[T,F,T]: level 0 has
    L = 32^3 = 32768 tokens, d = 64), 250-step DDIM (eta = 0), batch 1: the public generate(sampler='ddim') path (graph replay,
    device-resident timestep sequence) timed over a 16-step slice of the 250-step sequence, plus the flash attention kernel's
    roofline from per-launch events."""
    import types
    B, S, C, T, steps, K = 1, 32, 256, 1000, 250, 16
    dm = b200dm.DiffusionModel(S, 256, C, None, types.SimpleNamespace(timesteps=T, num_gpus=1, kernel_resize=False, bs=B))
    dm.network = b200dm.build_model(S, C, [64, 128, 256], [True, False, True])
    shape = (B, S, S, S, C)
    seq = list(range(T - 1, T - 1 - (T // steps) * K, -(T // steps)))   # the first K entries of the 250-step sequence 999, 995, ...
    lat = dm.generate(shape, seed=1, sampler="ddim", timestep_seq=seq)    # compile + capture
    flag = L.debug_flag()
    assert torch.isfinite(lat).all() and flag == 0, f"cfg-4: finite {bool(torch.isfinite(lat).all())}, watchdog flag {flag:#x}"
    ms = event_time(lambda: dm.generate(shape, seed=1, sampler="ddim", timestep_seq=seq), 2, 1)
    n_steps = len(seq)
    rows = dm._step["net"].prog.run_timed()
    attn = [r for r in rows if r[0] == "attn"]
    a_ms, a_fl = sum(r[3] for r in attn), sum(r[2] for r in attn)
    big = max(attn, key=lambda r: r[2])
    tens = [r for r in rows if r[0] in ("conv", "conv_halo", "attn")]
    return {"workload": "cfg-4: dm3d U-Net, has_attention=[T,F,T] (level-0 self-attention: L = 32768, d = 64), DDIM 250 of 1000 steps, batch 1",
            "ms_per_step": ms / n_steps, "steps_timed": n_steps, "volume_steps_per_s": B * n_steps / (ms * 1e-3),
            "seconds_per_250_step_chain": 250 * ms / n_steps * 1e-3,
            "call": "DiffusionModel.generate(shape, sampler='ddim', timestep_seq=<first 16 of the 250>) (graph replay; device-generated x_T)",
            "roofline_flash_attention": {"kernel": "flash_attn_kernel (tcgen05 QK^T / PV, online softmax, no (L, L) tensor)", "bound": "tensor",
                                         "achieved": a_fl / (a_ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                                         "frac": a_fl / (a_ms * 1e-3) / 1e12 / tf_peak, "launches": len(attn), "ms": a_ms,
                                         "largest_launch": {"op": big[1], "ms": big[3], "tflops": big[2] / (big[3] * 1e-3) / 1e12},
                                         "share_of_step": a_ms / sum(r[3] for r in rows)},
            "roofline_step": {"bound": "tensor", "algorithmic_gflop": sum(r[2] for r in tens) / 1e9,
                              "achieved": sum(r[2] for r in tens) / (ms / n_steps * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                              "frac": sum(r[2] for r in tens) / (ms / n_steps * 1e-3) / 1e12 / tf_peak}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sustained", action="store_true", help="skip the 1000-step sustained legs (tuning runs)")
    ap.add_argument("--no-cfg3", action="store_true", help="skip the cfg-3 (quantize + decode) leg (tuning runs)")
    ap.add_argument("--batch", type=int, default=None, help="tuning aid: per-GPU batch other than the cfg-2 value (8); not a bench line")
    ap.add_argument("--dump-ops", default=None, help="write per-op (kind,name,work,ms) CSV of one step")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the latents of the last timed step to DIR as float32 .npy (a fixed, seeded sample when larger than 32 MB)")
    args = ap.parse_args()
    if not 1 <= args.steps <= CFG["T"] - max(args.warmup, 3):
        ap.error(f"--steps must be in [1, {CFG['T']} - max(--warmup, 3)]: the timed steps walk one T={CFG['T']} timestep sequence")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's latents (--impl ours)")
    if args.batch:
        CFG["B"] = args.batch
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
