#!/usr/bin/env python
"""bench.py -- latent hot-path throughput on B200 (contract: one JSON line on stdout).

Workload (BASELINE.json configs[2] latent shape, the one the north_star's 70 %-of-HBM target is
quoted on): per step and per GPU, B = 4096 rows of the Clifford-torus latent at d = 2048
  1. fused Clifford power-spherical rsample + entropy/KL (device Philox RNG, one kappa per row)
     -> z (B, 4096)                                   [reference dists/clifford.py:295-327]
  2. vsa.bind(z, roles) with per-row roles (B, 4096)  [reference utils/vsa.py:43-46]
`value` = samples/s with inputs resident in HBM (two rotating buffer sets, 2 x 224 MB > 126 MB L2);
`e2e` = the same step through the reference-named Python API with HOST (pinned) inputs/outputs.
`--impl reference` times the reference's OWN classes on the host cores (staged copy under oracle/_ref, see
oracle/stage_reference.py; falls back to the oracle port only when no copy of the reference is available).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "clifford-vae_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

B_ROWS, D_LAT = 4096, 2048          # per GPU
N_VEC = 2 * D_LAT
METRIC = "latent rsample+KL+bind samples/s"
UNIT = "samples/s"
WORKLOAD = ("C3 latent: Clifford-PS fused rsample+KL (device RNG, row-scalar kappa) d=2048 -> z (4096 x 4096), "
            "then vsa.bind(z, roles) n=4096; B=4096 rows per GPU per step")
# algorithmic bytes per sample (SURVEY.md 8(d)): rsample+KL 12d+8, bind 12n
BYTES_RSAMPLE = 12 * D_LAT + 8
BYTES_BIND = 12 * N_VEC


TRAFFIC_FILE = "profiles/r02_traffic.json"


def load_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel.  ncu cannot run inside the timed
    bench, so the figure comes from the committed `ncu --set full` capture of this very command (profiles/README.md,
    regenerated with the kernels it describes); None when the file has no entry for the kernel."""
    try:
        with open(os.path.join(ROOT, TRAFFIC_FILE)) as f:
            t = json.load(f)
        for k, v in t.items():
            if kernel_name.startswith(k):
                return v["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own torch CPU path (oracle/_ref), else the oracle port
# --------------------------------------------------------------------------------------------------
REF_ROWS = 1024     # bounded sample of the 4096-row step (the reference runs at ~1e3 samples/s on 16 host threads)


def make_cpu_step(torch):
    """-> (step(loc, kap, roles) -> (bound, kl), kind, description).  kind "reference": the reference's classes,
    imported unmodified (dists/clifford.py:295-327 rsample + kl_divergence, utils/vsa.py:43-46 bind), constructed the
    way its conv VAE does (cnn/models.py:226-231: concentration expanded to loc's shape).  kind "port": the oracle
    restatement, used only when neither /root/reference nor oracle/_ref exists."""
    from oracle import reference_loader as RL
    ref = RL.load()
    if ref is not None:
        C, V = ref.clifford, ref.vsa
        prior = C.CliffordTorusUniform(D_LAT)

        def step(loc, kap, roles):
            q = C.CliffordPowerSphericalDistribution(loc, kap.expand_as(loc))
            z = q.rsample()
            kl = torch.distributions.kl.kl_divergence(q, prior)
            return V.bind(z, roles), kl
        return step, "reference", f"the reference's own classes ({ref.kind} copy), torch {torch.__version__} CPU"

    from oracle import latent_oracle as O

    def step(loc, kap, roles):
        rows, d = loc.shape
        alpha = 0.5 + kap + 1e-7
        tprime = torch.distributions.Beta(alpha.expand(rows, d), torch.full((rows, d), 0.5)).sample()
        g = torch.randn(rows, d)
        z = O.clifford_ps_rsample(loc, kap, tprime, g)
        kl = O.clifford_ps_kl(kap.expand(rows, d))
        return O.bind(z, roles), kl
    return step, "port", f"oracle port of the reference's torch CPU path, torch {torch.__version__} CPU"


def cpu_inputs(torch, rows):
    torch.manual_seed(0)
    loc = torch.randn(rows, D_LAT)
    kap = torch.rand(rows, 1) * 9.87 + 0.13
    roles = torch.randn(rows, N_VEC) / math.sqrt(N_VEC)
    return loc, kap, roles


def cpu_timing(rows, reps):
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind, desc = make_cpu_step(torch)
    loc, kap, roles = cpu_inputs(torch, rows)
    with torch.no_grad():
        step(loc, kap, roles)          # warm-up
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            step(loc, kap, roles)
            ts.append(time.perf_counter() - t0)
    return rows / statistics.median(ts), torch.get_num_threads(), ts, kind, desc


def bench_config():
    """`config` of both arms (identical keys and values: same workload, same shapes)."""
    return {"workload": WORKLOAD, "rows_per_gpu": B_ROWS, "d": D_LAT,
            "rng": "b200 arm: Philox4x32-10 on the device; reference arm: torch CPU generator",
            "l2": "b200 arm: inputs rotate over 2 buffer sets of 224 MB (> 126 MB L2)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind, desc = make_cpu_step(torch)
    rows = REF_ROWS
    loc, kap, roles = cpu_inputs(torch, rows)
    with torch.no_grad():
        for _ in range(args.warmup):
            step(loc, kap, roles)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step(loc, kap, roles)
        dt = time.perf_counter() - t0
    val = rows * args.steps / dt
    sample = f"{rows} of the {B_ROWS} rows per step (same d={D_LAT}); {desc}"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from clifford_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _lib.ensure_device(dev)
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    B, d, n = B_ROWS, D_LAT, N_VEC
    torch.manual_seed(1234 + rank)
    NSETS = 2
    sets = []
    for _ in range(NSETS):
        sets.append(dict(
            loc=torch.randn(B, d, device=dev), kap=(torch.rand(B, device=dev) * 9.87 + 0.13),
            roles=torch.randn(B, n, device=dev) / math.sqrt(n), z=torch.empty(B, n, device=dev),
            out=torch.empty(B, n, device=dev), kl=torch.empty(B, device=dev), ent=torch.empty(B, device=dev)))
    seed = 1234 + rank

    def step(i, ev=None):
        s = sets[i % NSETS]
        if ev:
            ev[0].record()
        rc = lib.cvb_clifford_ps_rsample(s["loc"].data_ptr(), s["kap"].data_ptr(), 1, 0, B, None, None, seed, i,
                                         s["z"].data_ptr(), None, s["ent"].data_ptr(), s["kl"].data_ptr(), None, B, d, st)
        if ev:
            ev[1].record()
        rc |= lib.cvb_vsa_bind(s["z"].data_ptr(), s["roles"].data_ptr(), s["out"].data_ptr(), B, B, B, n, 0, st)
        if ev:
            ev[2].record()
        if rc:
            raise RuntimeError(lib.cvb_last_error_string().decode())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    l0 = _lib.launch_count()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    for i in range(args.steps):
        step(args.warmup + i, evs[i])
    t_end.record()
    barrier()
    launches = _lib.launch_count() - l0
    ms_total = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:        # before the fused variant below overwrites the same buffers
        dump_outputs(args.dump_outputs, sets[(args.warmup + args.steps - 1) % NSETS])

    # the same outputs (z, KL, bound) from ONE launch (cvb_clifford_ps_rsample_bind: the sample's spectrum is known, so the
    # bind needs two transforms instead of three and z is not re-read) -- reported beside the headline, not as it
    def fused_step(i):
        s = sets[i % NSETS]
        rc = lib.cvb_clifford_ps_rsample_bind(s["loc"].data_ptr(), s["kap"].data_ptr(), B, None, None, seed, i,
                                              s["roles"].data_ptr(), B, s["z"].data_ptr(), s["out"].data_ptr(),
                                              s["ent"].data_ptr(), s["kl"].data_ptr(), None, B, d, st)
        if rc:
            raise RuntimeError(lib.cvb_last_error_string().decode())
    for i in range(3):
        fused_step(i)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(args.steps):
        fused_step(i)
    f1.record()
    barrier()
    ms_fused = f0.elapsed_time(f1) / args.steps
    ms_rs = sum(e[0].elapsed_time(e[1]) for e in evs) / args.steps
    ms_bind = sum(e[1].elapsed_time(e[2]) for e in evs) / args.steps

    # ---- e2e: reference-named Python API, host (pinned) buffers in and out ------------------------
    # One packed pinned buffer per direction: [loc | kappa | roles] in (one H2D copy per step), [bound | kl] out (one
    # D2H copy per step); the device tensors the API sees are views of the packed device buffers.
    from dists.clifford import CliffordPowerSphericalDistribution, CliffordTorusUniform
    from utils import vsa
    n_in, n_out = B * d + B + B * n, B * n + B
    h_in = torch.empty(n_in).pin_memory()
    h_in[:B * d].normal_()
    h_in[B * d:B * d + B].uniform_(0.13, 10.0)
    h_in[B * d + B:].normal_().mul_(1.0 / math.sqrt(n))
    h_out = torch.empty(n_out).pin_memory()
    prior = CliffordTorusUniform(d, device=dev)

    # Double-buffered pipeline: copy-in (H2D), compute, copy-out (D2H) on three streams, two device buffer
    # sets; every step still moves its own inputs from pinned host memory and its own results back.
    s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    dbuf = [dict(inp=torch.empty(n_in, device=dev), out=torch.empty(n_out, device=dev),
                 ev_in=torch.cuda.Event(), ev_cmp=torch.cuda.Event(), ev_out=torch.cuda.Event()) for _ in range(2)]

    def e2e_step(i, compute=True):
        b = dbuf[i % 2]
        with torch.no_grad():
            with torch.cuda.stream(s_in):
                s_in.wait_event(b["ev_cmp"])                  # the compute that last read this set is done
                b["inp"].copy_(h_in, non_blocking=True)
                b["ev_in"].record(s_in)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(b["ev_in"])
                s_cmp.wait_event(b["ev_out"])                 # the previous outputs of this set were copied out
                if compute:
                    loc_v = b["inp"][:B * d].view(B, d)
                    kap_v = b["inp"][B * d:B * d + B].view(B, 1)
                    roles_v = b["inp"][B * d + B:].view(B, n)
                    q = CliffordPowerSphericalDistribution(loc_v, kap_v, validate_args=False)
                    z = q.rsample()
                    kl = torch.distributions.kl.kl_divergence(q, prior)
                    bound = vsa.bind(z, roles_v)
                    b["out"][:B * n].view(B, n).copy_(bound)      # the API allocates its result; gather it next to kl
                    b["out"][B * n:].copy_(kl)
                b["ev_cmp"].record(s_cmp)
            with torch.cuda.stream(s_out):
                s_out.wait_event(b["ev_cmp"])
                h_out.copy_(b["out"], non_blocking=True)
                b["ev_out"].record(s_out)

    def e2e_drain():
        s_in.synchronize(); s_cmp.synchronize(); s_out.synchronize()

    def e2e_time(steps, compute):
        for i in range(4):
            e2e_step(i, compute)
        e2e_drain()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s_in.wait_event(e0); s_cmp.wait_event(e0); s_out.wait_event(e0)
        for i in range(steps):
            e2e_step(i, compute)
        e2e_drain()
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    e2e_steps = max(3, min(args.steps, 20))
    ms_e2e = e2e_time(e2e_steps, True)
    # the link ceiling on this box: the same two copies per step (full duplex) with no kernel in between
    ms_link = e2e_time(e2e_steps, False)
    clk = clocks.stop() if rank == 0 else None

    vae = None if args.no_vae_step else vae_train_leg(torch, dev, world, rank, local)
    peak, peak_src = load_peaks()
    other = None
    if not args.no_other_configs:
        other = reduce_legs(torch, dist, config_legs(torch, lib, dev, st, world), dev, world, peak)

    # max over ranks
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e, ms_rs, ms_bind, ms_link, ms_fused], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e, ms_rs, ms_bind, ms_link, ms_fused = (float(x) for x in t.tolist())

    if rank == 0:
        value = world * B * args.steps / (ms_total * 1e-3)
        e2e_val = world * B * e2e_steps / (ms_e2e * 1e-3)
        k_rs = {"name": "clifford_fwd_kernel<11,PsRng,rowk>", "ms": ms_rs, "bytes": B * BYTES_RSAMPLE}
        k_bd = {"name": "bind_v3_kernel<11,Mul,direct>", "ms": ms_bind, "bytes": B * BYTES_BIND}
        dom = k_rs if ms_rs >= ms_bind else k_bd
        achieved = dom["bytes"] / (dom["ms"] * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": bench_config(),
            "roofline": {"bound": "hbm", "kernel": dom["name"], "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": load_traffic(dom["name"]),
                         "traffic_source": f"{TRAFFIC_FILE}: static, from the committed ncu --set full capture of this command",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": dom["bytes"], "ms_per_launch": dom["ms"]},
            "kernels": {
                "rsample_kl": {"ms": ms_rs, "GBps": k_rs["bytes"] / (ms_rs * 1e-3) / 1e9,
                               "frac": k_rs["bytes"] / (ms_rs * 1e-3) / 1e9 / peak},
                "bind": {"ms": ms_bind, "GBps": k_bd["bytes"] / (ms_bind * 1e-3) / 1e9,
                         "frac": k_bd["bytes"] / (ms_bind * 1e-3) / 1e9 / peak},
                "fused_one_launch_variant": {
                    "what": "cvb_clifford_ps_rsample_bind: z, KL and bind(z, roles) from one kernel (28d+12 B per row)",
                    "ms": ms_fused, "samples_per_s": world * B / (ms_fused * 1e-3),
                    "GBps": B * (28 * d + 12) / (ms_fused * 1e-3) / 1e9,
                    "frac": B * (28 * d + 12) / (ms_fused * 1e-3) / 1e9 / peak}},
            "e2e": {"value": e2e_val, "unit": UNIT, "steps": e2e_steps,
                    "h2d_bytes_per_step": world * n_in * 4, "d2h_bytes_per_step": world * n_out * 4,
                    "api": "dists.clifford.CliffordPowerSphericalDistribution.rsample + kl_divergence + utils.vsa.bind",
                    "pipeline": "double-buffered: one packed H2D copy [loc|kappa|roles], compute, one packed D2H copy "
                                "[bound|kl] per step on three streams",
                    "link_ceiling": {"value": world * B * e2e_steps / (ms_link * 1e-3), "unit": UNIT,
                                     "h2d_GBps_per_gpu": n_in * 4 * e2e_steps / (ms_link * 1e-3) / 1e9,
                                     "d2h_GBps_per_gpu": n_out * 4 * e2e_steps / (ms_link * 1e-3) / 1e9,
                                     "what": "the same pinned copies per step with no kernel between them, all ranks at once "
                                             "(max over ranks): what the host link of this box allows"},
                    "frac_of_link_ceiling": ms_link / ms_e2e},
            "gpu_launches": int(launches), "clocks": clk,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, cores, ts, kind, desc = cpu_timing(REF_ROWS, 5)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": f"{REF_ROWS} of the {B} rows (same d={d}), median of 5 passes "
                                              f"({sum(ts):.1f} s CPU); {desc}"}
        if vae is not None:
            line["vae_train_step"] = vae
        if other is not None:
            line["other_configs"] = other
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_ROWS = 1024    # rows of z and of bind(z, roles) written by --dump-outputs: 2 x 16 MB of the 2 x 64 MB


def dump_outputs(out_dir, s):
    """Write what the last timed step returned as float32 .npy files: z and bind(z, roles) on a fixed, seeded sample of
    DUMP_ROWS rows (ascending row order), KL and entropy for every row.  The inputs and the device RNG are seeded, so
    two builds run with the same arguments can be compared file for file."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rows = torch.randperm(B_ROWS, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    rows = rows.to(s["z"].device)
    arrays = {"z": s["z"].index_select(0, rows), "bound": s["out"].index_select(0, rows), "kl": s["kl"],
              "entropy": s["ent"]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def vae_train_leg(torch, dev, world, rank, local, steps=8, warmup=3, compare_reference_dists=True):
    """Second half of BASELINE.json's metric: the C3 training step of the reference's OWN model -- `cnn.models.VAE(
    latent_dim=2048, in_channels=3, distribution="clifford", device, recon_loss_type="l1")` (cnn/models.py:134-315,
    18.4 M parameters), loaded unmodified from the staged copy under oracle/_ref with `dists.clifford` resolved to the
    drop-in classes -- run the way cnn/cifar10_train.py:62-77 runs it (zero_grad, forward, compute_loss, backward,
    clip_grad_norm_ 1.0, AdamW lr 3e-4 step; the per-step .item() logging left out), batch 4096 per GPU, synthetic
    U(-1,1) 3x32x32 inputs, DistributedDataParallel over NCCL when world > 1.  Every rank runs it; the time is the
    max over ranks.  At world == 1 the same step is also timed with the reference's own distribution classes on the
    GPU (eager PyTorch + cuFFT): the "reference on cuda" comparator of BASELINE.md.  Falls back to the stand-in conv
    VAE of examples/train_vae_ddp.py only when no copy of the reference is available."""
    import torch.distributed as dist
    import torch.nn as nn
    import importlib.util
    spec = importlib.util.spec_from_file_location("train_vae_ddp", os.path.join(ROOT, "examples", "train_vae_ddp.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    from oracle import reference_loader as RL
    ref = RL.load()
    batch = 4096
    torch.manual_seed(1234 + rank)

    def reference_model_step(models_mod):
        model = models_mod.VAE(latent_dim=D_LAT, in_channels=3, distribution="clifford", device=dev, recon_loss_type="l1")
        net = nn.parallel.DistributedDataParallel(model, device_ids=[local]) if world > 1 else model
        opt = torch.optim.AdamW(net.parameters(), lr=3e-4)
        x = torch.rand(batch, 3, 32, 32, device=dev) * 2 - 1

        def step():
            opt.zero_grad()
            x_recon, q_z, p_z, _ = net(x)
            losses = model.compute_loss(x, x_recon, q_z, p_z, 1.0)
            losses["total_loss"].backward()
            torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
            opt.step()
            return losses["total_loss"]
        return step, sum(p.numel() for p in model.parameters())

    out = {"batch_per_gpu": batch, "n_gpus": world, "parallelism": f"ddp{world}" if world > 1 else "single",
           "steps": steps, "warmup": warmup}
    if ref is not None:
        step, nparam = reference_model_step(RL.models(ref, "cnn"))
        out["model"] = (f"reference cnn.models.VAE(latent_dim={D_LAT}, in_channels=3, distribution='clifford', "
                        f"recon_loss_type='l1') [{ref.kind} copy, unmodified], {nparam} parameters, AdamW lr 3e-4, clip 1.0; "
                        "dists.clifford = drop-in kernels")
    else:
        step = mod.make_training_step("conv", "clifford", D_LAT, batch, dev, world, local)
        out["model"] = "stand-in conv VAE (examples/train_vae_ddp.py): no copy of the reference available"
    ms, loss = mod.time_training_steps(step, steps, warmup, dev, world)
    out.update({"ms_per_step": ms, "steps_per_s": 1e3 / ms, "samples_per_s": world * batch * 1e3 / ms, "loss": loss})
    del step
    torch.cuda.empty_cache()
    if ref is not None and world == 1 and compare_reference_dists:
        try:
            step, _ = reference_model_step(RL.models(ref, "cnn", ref.clifford))
            ms_r, loss_r = mod.time_training_steps(step, max(3, steps // 2), 2, dev, world)
            out["reference_on_cuda"] = {"what": "same model and step with the reference's own dists/clifford.py classes "
                                                "on the GPU (eager PyTorch, cuFFT, torch._sample_dirichlet)",
                                        "ms_per_step": ms_r, "steps_per_s": 1e3 / ms_r, "loss": loss_r,
                                        "speedup_of_drop_in": ms_r / ms}
            del step
        except Exception as e:          # the comparator must never take the bench line down
            out["reference_on_cuda"] = {"error": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    return out


def config_legs(torch, lib, dev, st, world):
    """The other BASELINE.json configurations at their stated sizes, every rank on its own shard (weak scaling, no
    data-path collective); returns [(name, info dict, local ms)], the caller reduces the times with MAX over ranks.
      C1  Clifford rsample+KL  B=128  d=512 (one launch)          C2  PowerSpherical / vMF rsample+KL  B=1024  D=513
      C3  rsample backward and log_prob at B=4096 d=2048          C4  bind / unbind sweep, 2^20 vectors per GPU, d=1024..16384
      C5  depth-1..32 bind -> reverse unbind -> cosine, d=8192, 512 trials per depth per GPU (fused chain kernel)"""
    from clifford_b200 import harness
    from utils import vsa
    legs = []

    def timeit(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    # ---- C4: 2^20 vectors per GPU, streamed in chunks of <= 12 GiB working set (d = 16384 would need 192 GiB at once)
    NV = 1 << 20
    for dd in (1024, 2048, 4096, 8192, 16384):
        chunk = min(NV, (12 << 30) // (12 * dd))
        chunk = 1 << (chunk.bit_length() - 1)
        a = torch.randn(chunk, dd, device=dev)
        b = torch.randn(chunk, dd, device=dev)
        o = torch.empty(chunk, dd, device=dev)
        nchunks = NV // chunk
        modes = (("bind", 0), ("unbind_inv", 1), ("unbind_deconv", 2)) if dd in (1024, 4096, 16384) else (("bind", 0),)
        for opname, mode in modes:
            def run(mode=mode):
                for _ in range(nchunks):
                    lib.cvb_vsa_bind(a.data_ptr(), b.data_ptr(), o.data_ptr(), chunk, chunk, chunk, dd, mode, st)
            ms = timeit(run, reps=2, warm=1)
            legs.append((f"C4_{opname}_d{dd}", {"vectors_per_gpu": NV, "chunk": chunk, "unit": "vec/s", "units": NV,
                                                "bytes_per_unit": 12 * dd}, ms))
        if dd == 4096:
            out1 = torch.empty(chunk, device=dev)
            ms = timeit(lambda: [lib.cvb_vsa_cosine(a.data_ptr(), b.data_ptr(), out1.data_ptr(), chunk, chunk, chunk, dd, st)
                                 for _ in range(nchunks)], reps=2, warm=1)
            legs.append((f"C4_similarity_d{dd}", {"vectors_per_gpu": NV, "chunk": chunk, "unit": "pairs/s", "units": NV,
                                                  "bytes_per_unit": 8 * dd + 4}, ms))
            ws = torch.empty(max(int(lib.cvb_vsa_bundle_workspace_bytes(chunk, dd)) // 4, 1), device=dev)
            outv = torch.empty(dd, device=dev)
            ms = timeit(lambda: [lib.cvb_vsa_bundle(a.data_ptr(), outv.data_ptr(), chunk, dd, 1.0, ws.data_ptr(), st)
                                 for _ in range(nchunks)], reps=2, warm=1)
            legs.append((f"C4_bundle_d{dd}", {"vectors_per_gpu": NV, "chunk": chunk, "unit": "vec/s", "units": NV,
                                              "bytes_per_unit": 4 * dd}, ms))
            del out1, ws, outv
        del a, b, o
    torch.cuda.empty_cache()

    # ---- C3: the rest of the training path at the headline shape
    B, d = B_ROWS, D_LAT
    loc = torch.randn(B, d, device=dev)
    kap = torch.rand(B, device=dev) * 9.87 + 0.13
    z = torch.empty(B, 2 * d, device=dev)
    tps = torch.empty(B, d, device=dev)
    gz = torch.randn(B, 2 * d, device=dev)
    dloc = torch.empty(B, d, device=dev)
    dk = torch.empty(B, device=dev)
    lp = torch.empty(B, device=dev)
    lib.cvb_clifford_ps_rsample(loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, 7, 0, z.data_ptr(), tps.data_ptr(),
                                None, None, None, B, d, st)
    flush = torch.empty(64 << 20, device=dev)          # 256 MB > L2: written between repetitions

    def with_flush(fn):
        def run():
            flush.zero_()
            fn()
        return run
    ms_flush = timeit(lambda: flush.zero_(), reps=10)
    ms = timeit(with_flush(lambda: lib.cvb_clifford_ps_rsample_backward(
        gz.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, None, None, tps.data_ptr(), dloc.data_ptr(),
        dk.data_ptr(), B, d, st)), reps=10) - ms_flush
    legs.append(("C3_rsample_backward_B4096_d2048", {"rows": B, "unit": "samples/s", "units": B, "bytes_per_unit": 20 * d + 8,
                                                     "l2": "256 MB flush between repetitions (its time subtracted)"}, ms))
    ms = timeit(with_flush(lambda: lib.cvb_clifford_ps_log_prob(
        z.data_ptr(), loc.data_ptr(), kap.data_ptr(), 1, 0, B, lp.data_ptr(), None, None, None, B, d, st)), reps=10) - ms_flush
    legs.append(("C3_log_prob_B4096_d2048", {"rows": B, "unit": "samples/s", "units": B, "bytes_per_unit": 12 * d + 8,
                                             "l2": "256 MB flush between repetitions (its time subtracted)"}, ms))
    del loc, z, tps, gz, dloc

    # ---- C1 / C2: launch-latency-sized configurations
    B1, d1 = 128, 512
    loc1 = torch.randn(B1, d1, device=dev)
    kap1 = torch.rand(B1, device=dev) * 9.97 + 0.03
    z1 = torch.empty(B1, 2 * d1, device=dev)
    kl1 = torch.empty(B1, device=dev)
    ms = timeit(lambda: lib.cvb_clifford_ps_rsample(loc1.data_ptr(), kap1.data_ptr(), 1, 0, B1, None, None, 7, 0, z1.data_ptr(),
                                                    None, None, kl1.data_ptr(), None, B1, d1, st), reps=50)
    legs.append(("C1_clifford_rsample_kl_B128_d512", {"rows": B1, "unit": "samples/s", "units": B1,
                                                      "bytes_per_unit": 12 * d1 + 8, "launches_per_step": 1}, ms))
    B2, D2 = 1024, 513
    loc = torch.nn.functional.normalize(torch.randn(B2, D2, device=dev), dim=-1)
    kap2 = torch.rand(B2, device=dev) * 9.2 + 0.8
    z = torch.empty(B2, D2, device=dev)
    save = torch.empty(B2, 2, device=dev)
    ent = torch.empty(B2, device=dev)
    kl = torch.empty(B2, device=dev)

    # rsample fused with entropy / KL: ONE launch per step (round 1: sampler + entropy kernel)
    def ps_step():
        lib.cvb_powerspherical_rsample_kl(loc.data_ptr(), kap2.data_ptr(), B2, None, None, 3, 0, z.data_ptr(), save.data_ptr(),
                                          ent.data_ptr(), kl.data_ptr(), None, B2, D2, st)

    def vmf_step():
        lib.cvb_vmf_rsample_kl(loc.data_ptr(), kap2.data_ptr(), B2, None, None, 0, None, 3, 0, z.data_ptr(), save.data_ptr(),
                               ent.data_ptr(), kl.data_ptr(), None, None, None, B2, D2, st)

    for name, fn in (("C2_powerspherical_rsample_kl_B1024_D513", ps_step), ("C2_vmf_rsample_kl_B1024_D513", vmf_step)):
        ms = timeit(fn, reps=50)
        legs.append((name, {"rows": B2, "unit": "samples/s", "units": B2, "bytes_per_unit": 8 * D2 + 8,
                            "launches_per_step": 1, "note": "4 MB per step: launch-latency bound at this batch"}, ms))

    # the same C1 / C2 steps captured once in a CUDA graph and replayed (device-resident Philox launch counter, so every
    # replay draws a fresh stream: cvb_set_rng_device_counter_autobump -- the sampling kernel bumps the counter itself)
    ctr = torch.zeros(1, dtype=torch.int64, device=dev)
    lib.cvb_set_rng_device_counter_autobump(ctr.data_ptr())   # self-bumping: no counter-increment kernel between the steps

    def cur():
        return torch.cuda.current_stream().cuda_stream

    def g_c1():
        lib.cvb_clifford_ps_rsample(loc1.data_ptr(), kap1.data_ptr(), 1, 0, B1, None, None, 7, 0, z1.data_ptr(), None, None,
                                    kl1.data_ptr(), None, B1, d1, cur())

    def g_ps():
        lib.cvb_powerspherical_rsample_kl(loc.data_ptr(), kap2.data_ptr(), B2, None, None, 3, 0, z.data_ptr(), save.data_ptr(),
                                          ent.data_ptr(), kl.data_ptr(), None, B2, D2, cur())

    def g_vmf():
        lib.cvb_vmf_rsample_kl(loc.data_ptr(), kap2.data_ptr(), B2, None, None, 0, None, 3, 0, z.data_ptr(), save.data_ptr(),
                               ent.data_ptr(), kl.data_ptr(), None, None, None, B2, D2, cur())

    for name, fn, rows, bpu in (("C1_clifford_rsample_kl_B128_d512_graph", g_c1, B1, 12 * d1 + 8),
                                ("C2_powerspherical_rsample_kl_B1024_D513_graph", g_ps, B2, 8 * D2 + 8),
                                ("C2_vmf_rsample_kl_B1024_D513_graph", g_vmf, B2, 8 * D2 + 8)):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(10):                 # ten steps per replay: the replay launch cost is amortised like a training loop's
                fn()
        ms = timeit(graph.replay, reps=20) / 10
        legs.append((name, {"rows": rows, "unit": "samples/s", "units": rows, "bytes_per_unit": bpu,
                            "note": "CUDA graph of 10 steps replayed; fresh draws per replay"}, ms))
    lib.cvb_set_rng_device_counter_autobump(None)
    assert int(ctr.item()) > 0                 # the kernels really bumped it

    # ---- C5: depth 1..32 at d = 8192, 512 trials per depth per GPU, whole chain + cosine in one kernel per depth
    d5, T5, depths = 8192, 512, list(range(1, 33))
    pool = vsa.normalize_vectors(vsa.unitary_init(T5 * 33, d5, device=dev))

    def c5():
        sims = []
        for m in depths:
            sims.append(harness.binding_depth_cell_fused(pool[:T5 * (m + 1)].view(T5, m + 1, d5)).mean())
        return torch.stack(sims)
    sims = c5()
    ms = timeit(c5, reps=2, warm=1)
    ops = T5 * sum(2 * m for m in depths)
    legs.append(("C5_depth_1_32_d8192", {"trials_per_depth_per_gpu": T5, "unit": "bind+unbind ops/s", "units": ops,
                                         "bytes_per_unit": None, "algorithmic_bytes": sum(4 * d5 * (m + 1) * T5 for m in depths),
                                         "min_similarity_unitary_keys": float(sims.min())}, ms))
    return legs


def reduce_legs(torch, dist, legs, dev, world, peak):
    """MAX over ranks of every leg's time; aggregate throughput = world * units / time."""
    t = torch.tensor([ms for _, _, ms in legs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = {}
    for (name, info, _), ms in zip(legs, t.tolist()):
        e = dict(info)
        units = e.pop("units")
        e["ms"] = ms
        e["n_gpus"] = world
        e["per_s"] = world * units / (ms * 1e-3)
        if e.get("bytes_per_unit"):
            gb = units * e["bytes_per_unit"] / (ms * 1e-3) / 1e9
            e["GBps_per_gpu"] = gb
            e["frac"] = gb / peak
        elif e.get("algorithmic_bytes"):
            gb = e["algorithmic_bytes"] / (ms * 1e-3) / 1e9
            e["GBps_per_gpu"] = gb
            e["frac"] = gb / peak
        out[name] = e
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-other-configs", action="store_true", help="skip the C1/C2/C3-bwd/C4/C5 legs (other_configs)")
    ap.add_argument("--no-vae-step", action="store_true", help="skip the C3 VAE training-step leg (vae_train_step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's z, bind(z, roles) (seeded sample of rows), KL and "
                         "entropy to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
