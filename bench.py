"""bench.py — vectors quantized / second at dim=256, codebook=1024 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2|cfg5] [--dump-outputs DIR]

Workload (N=1 and per GPU for N>1): BASELINE.json configs[1] — VectorQuantize(dim=256, codebook_size=1024),
x = (64, 4096, 256) bf16, training-mode forward with the EMA codebook update.  A "step" is one such
forward over one synthetic batch.  `value` times the device-resident path with CUDA events; `e2e` times
the public module call with HOST (pinned) buffers, host<->device copies inside the timed region.
Under torchrun every rank runs the same per-GPU batch (weak scaling) with sync_codebook=True: the packed EMA
statistics are summed over the ranks inside the EMA kernels (NVLink peer loads from symmetric memory after one
barrier kernel; ONE NCCL all-reduce if symmetric memory is unavailable); the time is the max over ranks.

`--impl reference` times the UNMODIFIED reference package (baseline/_ref) on the host cores — its own
VectorQuantize(dim=256, codebook_size=1024) training-mode forward on the full 262144-vector batch — and falls back
to the torch-CPU oracle port (oracle/vq_oracle_torch.py, the same ATen op sequence) only if the package cannot be
imported, saying so in `cpu_baseline.kind`.

`--dump-outputs DIR` writes what the last headline-timed step returned (rank 0's shard under torchrun) as float32 .npy
files: `indices` and `loss` whole, and `quantize_rows`, a fixed seeded sample of the quantized rows (their row numbers in
`quantize_row_ids`, float64).  Inputs and codebooks are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vectors quantized/sec at dim=256, codebook=1024; indices bit-exact vs ref"
B, T, D, K = 64, 4096, 256, 1024
WORKLOAD = "VectorQuantize dim=256 codebook_size=1024, x=(64,4096,256) bf16, EMA on (BASELINE.json configs[1])"
E2E_CHUNKS = int(os.environ.get("VQB_E2E_CHUNKS", "10"))  # row chunks of the host-buffer pipeline (forward_host)
DUMP_ROWS = 16384   # quantized rows sampled by --dump-outputs: 16 MB at D=256 in float32 (all of q would be 256 MB)


def dump_outputs(out_dir, q, ind, loss):
    """Write one step's outputs to out_dir as .npy: indices and loss whole, a fixed seeded sample of the quantized rows."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rows = q.detach().reshape(-1, q.shape[-1])
    pick = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    arrays = {"quantize_rows": rows[pick.to(rows.device)].float(), "quantize_row_ids": pick.double(),
              "indices": ind.float(),   # exact: codebook indices are far below 2**24
              "loss": loss.detach().float()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (reference algorithm on the host cores)
# ------------------------------------------------------------------------------------------------

CPU_THREADS = [None]
CPU_KIND = ["port"]
CPU_FULL_BATCH = (B, T)          # the reference arm runs the WHOLE config-2 batch per step (262144 vectors)


def cpu_reference_step_factory(threads=None):
    """One training-mode forward of the reference on the host cores, on the full BASELINE config-2 batch.

    Preferred: the UNMODIFIED reference package (`baseline/_ref`, pip-installed from /root/reference; `oracle/ref_loader.py`)
    through its own public API — `VectorQuantize(dim=256, codebook_size=1024)(x)` — kind "reference".  If it cannot be
    imported on this box: the torch-CPU oracle port (the same ATen op sequence, bit-identical on the goldens), kind "port"."""
    import torch
    torch.set_num_threads(threads or os.cpu_count())
    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(CPU_FULL_BATCH[0], CPU_FULL_BATCH[1], D, generator=gen).bfloat16()
    e = torch.randn(K, D, generator=gen)
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import ref_loader
        ref = ref_loader.load_reference()
        # sync_codebook=False: under torchrun the reference would otherwise all-reduce its CPU statistics over NCCL
        # (vqp:925-926); a single process owns this arm (rank 0), the arithmetic is the same
        vq = ref.VectorQuantize(dim=D, codebook_size=K, sync_codebook=False)
        with torch.no_grad():
            vq._codebook.embed.copy_(e[None]); vq._codebook.embed_avg.copy_(e[None])
        vq.train()
        CPU_KIND[0] = "reference"

        def step():
            with torch.no_grad():
                vq(x)
        return step
    except Exception as ex:  # noqa: BLE001 — any import problem falls back to the port, and the line says so
        sys.stderr.write(f"bench.py: reference package not importable ({ex!r}); timing the oracle port instead\n")
    from oracle import vq_oracle_torch as T  # the reference's own ATen op sequence (bit-identical on the goldens)
    state = T.State(e)
    CPU_KIND[0] = "port"

    def step():
        T.vq_forward(x, state, training=True)

    return step


def time_cpu(steps, warmup):
    """All host cores is torch's default (and what the reference would use); on many-core hosts a smaller pool is
    faster for this GEMM size, so both are timed and the FASTER one is reported (its thread count in `cores`)."""
    best = None
    n_vec = CPU_FULL_BATCH[0] * CPU_FULL_BATCH[1]
    for threads in sorted({os.cpu_count(), min(32, os.cpu_count())}, reverse=True):
        step = cpu_reference_step_factory(threads)
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
        cand = (n_vec * steps / dt, dt / steps * 1e3, threads)
        if best is None or cand[0] > best[0]:
            best = cand
    CPU_THREADS[0] = best[2]
    return best[0], best[1]


def cpu_baseline_block(value):
    what = ("the UNMODIFIED reference package (baseline/_ref), VectorQuantize(dim=256, codebook_size=1024) training-mode forward on CPU"
            if CPU_KIND[0] == "reference" else
            "oracle/vq_oracle_torch.py (the reference's ATen op sequence: N x K fp32 distances, one-hot, 3 sgemm)")
    return {"value": value, "unit": "vectors/s", "cores": CPU_THREADS[0] or os.cpu_count(), "host_cores": os.cpu_count(),
            "kind": CPU_KIND[0],
            "sample": f"the full {CPU_FULL_BATCH[0] * CPU_FULL_BATCH[1]}-vector batch of one step per CPU step; {what}; "
                      f"best of torch threads in {{all host cores, 32}}"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 for its workers; the reference arm is entitled to every host thread
    for var in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(var, None)
    steps = args.steps
    warm = max(1, min(args.warmup, 2))
    v, ms = time_cpu(steps, warm)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "vectors/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
        "cpu_baseline": cpu_baseline_block(v),
        "e2e": {"value": v, "unit": "vectors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks line")
# ------------------------------------------------------------------------------------------------

NCU_SUMMARY = "r2_assign_benched_summary.txt"   # ncu --set full of the search launch as benched (scripts/r2_profile.sh)


def ncu_dram_bytes():
    """dram read + write bytes of one vq_assign_kernel launch, from the committed ncu summary (None if it is missing)."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", NCU_SUMMARY)
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, seen = 0.0, 0
    try:
        for line in open(path):
            if "dram__bytes_read.sum =" in line or "dram__bytes_write.sum =" in line:
                val, unit = line.split("=")[1].split()[:2]
                total += float(val) * mult[unit]
                seen += 1
    except Exception:
        return None
    return total if seen == 2 else None


def pin_to_gpu_numa_node(local):
    """Bind this rank (and its pinned host buffers, by first touch) to the NUMA node its GPU hangs off: with 8 ranks
    pushing 270 MB per step each through host memory, remote-node traffic halves the e2e rate (round-1 SCALE: 0.57)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:  # noqa: BLE001 — topology files missing: leave the affinity alone
        pass
    return None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region, in-process through NVML.

    A forked `nvidia-smi -lms` loop was measured to perturb the very region it watches: one query can hold a driver lock
    for tens of milliseconds, and a 20-step timed region is only ~7 ms long (observed: 0.34 -> 1.5 / 3.1 ms per step when
    a query landed inside it).  NVML calls from a thread cost microseconds and fork nothing.
    """
    PERIOD_S = 0.002

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []          # (time, sm_mhz, reasons bitmask, power W)
        self.smax = None
        self.handle = None
        self.stop_flag = False
        self.thread = None
        self.nv = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes torch's visible devices; honour CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis:
                parts = [v.strip() for v in vis.split(",") if v.strip()]
                if self.gpu < len(parts) and parts[self.gpu].isdigit():
                    idx = int(parts[self.gpu])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                except Exception:
                    pw = None
                self.rows.append((time.time(), sm, rs, pw))
            except Exception:
                pass
            time.sleep(self.PERIOD_S)

    def stop(self, t0, t1):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        nv = self.nv
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                 ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                 ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        if not inside:  # the timed region was shorter than one sample period: take the nearest samples
            inside = sorted(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:3]
        sm = [r[1] for r in inside]
        reasons = sorted({n for r in inside for n, bit in names if r[2] & bit})
        pw = [r[3] for r in inside if r[3] is not None]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.smax, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "source": "nvml, in-process, 2 ms period"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    import vector_quantize_pytorch_b200 as vqb
    from vector_quantize_pytorch_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa_node(local)   # before any pinned allocation (first touch decides the node)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg5 = args.workload == "cfg5"
    torch.manual_seed(1234)  # same codebook on every rank (replicas)
    if cfg5:
        # BASELINE.json configs[4]: the GLOBAL batch (64, 4096, 256) is split over the ranks (strong scaling)
        assert B % world == 0
        b_local, in_dtype = B // world, torch.float32
        module = vqb.GroupedResidualVQ(dim=D, groups=2, num_quantizers=8, codebook_size=K, sync_codebook=world > 1).to(dev)
        books = [l._codebook for r in module.rvqs for l in r.layers]
        workload = ("GroupedResidualVQ dim=256 groups=2 num_quantizers=8 codebook_size=1024, global x=(64,4096,256) fp32 sharded on "
                    "batch, EMA on (BASELINE.json configs[4])")
    else:
        b_local, in_dtype = B, torch.bfloat16
        module = vqb.VectorQuantize(dim=D, codebook_size=K, sync_codebook=world > 1).to(dev)
        books = [module._codebook]
        workload = WORKLOAD
    with torch.no_grad():
        for cb in books:
            e = torch.randn(1, K, cb.dim, device=dev)
            cb.embed.copy_(e)
            cb.embed_avg.copy_(e)
    module.train()
    vq = module
    gen = torch.Generator().manual_seed(1234 + rank)  # every rank its own shard of the global batch
    x_host = torch.randn(b_local, T, D, generator=gen).to(in_dtype).pin_memory()
    x_dev = x_host.to(dev)
    n_vec = b_local * T

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---------------- device-resident timing (`value`)
    # W untimed warm-up steps as requested, plus enough extra untimed calls for the allocator / graph cache to reach
    # their steady state (every output-pointer set is enqueued directly once and captured once before it replays)
    for _ in range(max(args.warmup, 12)):
        q, ind, loss = vq(x_dev)   # same binding pattern as the timed loop: the allocator then cycles the same blocks
    barrier()
    ops.PROFILE_EVENTS = None
    ops.LAUNCHES = 0
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.05)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start = time.time()
    e0.record()
    for _ in range(args.steps):
        q, ind, loss = vq(x_dev)
    t_host = time.time()
    e1.record()
    barrier()
    t_end = time.time()
    launches = ops.LAUNCHES
    clocks = sampler.stop(t_start, t_end)
    ms_dev = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    host_ms = (t_host - t_start) * 1e3 / args.steps   # CPU time to enqueue one step (must stay below ms_dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, q, ind, loss)

    # ---------------- the dominant kernel's launch duration (roofline): the same K steps once more, now with a CUDA
    # event pair recorded on the launching stream around vq_assign_kernel.  Kept out of the headline region because
    # event records cannot live inside the step's CUDA graph: with them every launch of the chain is enqueued one by
    # one and the step becomes sensitive to host jitter (observed 0.34 -> 1.1 ms on a noisy box).
    def timed_loop(n_steps=None, seconds=None, events=False):
        """(ms per step, mean search-kernel ms or None, steps run, clocks record) of a loop of whole steps."""
        ops.PROFILE_EVENTS = [] if events else None
        smp = ClockSampler(local)
        smp.start()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        w0 = time.time()
        g0.record()
        done = 0
        while True:
            for _ in range(n_steps or 50):
                vq(x_dev)
            done += n_steps or 50
            if seconds is None:
                break
            if done % 500 == 0:
                torch.cuda.synchronize()   # keep the launch queue bounded; ~0.1 % of the loop
            if time.time() - w0 >= seconds:
                break
        g1.record()
        barrier()
        w1 = time.time()
        prof = [pr for pr in (ops.PROFILE_EVENTS or []) if pr is not None]
        ops.PROFILE_EVENTS = None
        kms = statistics.mean(a.elapsed_time(b) for a, b in prof) if prof else None
        return g0.elapsed_time(g1) / done, kms, done, smp.stop(w0, w1)

    ms_dev_events, assign_ms, _, _ = timed_loop(n_steps=args.steps, events=True)

    # ---------------- sustained block: the burst figures above come from a few milliseconds at boost clocks; the same step
    # looped for >= 2 s shows what the part sustains (clocks / power recorded), once replaying the step's graph (ms per step)
    # and once with the event pair around the search kernel (its duration under sustained clocks).
    sustained = None
    if not args.no_sustained and world == 1:
        s_ms, _, s_steps, s_clk = timed_loop(seconds=args.sustained_seconds)
        _, s_kms, _, s_clk2 = timed_loop(seconds=args.sustained_seconds, events=True)
        sustained = {"seconds": args.sustained_seconds, "steps": s_steps, "ms_per_step": s_ms,
                     "value": n_vec / (s_ms * 1e-3), "kernel_ms": s_kms, "clocks": s_clk, "clocks_event_loop": s_clk2}

    # ---------------- end-to-end timing (`e2e`): pinned host input -> module -> host outputs
    e2e = None
    if not cfg5 and not os.environ.get("VQB_BENCH_SKIP_E2E"):
        q_host = torch.empty((B, T, D), dtype=torch.bfloat16).pin_memory()
        i_host = torch.empty((B, T), dtype=torch.int64).pin_memory()
        l_host = torch.empty((), dtype=torch.float32).pin_memory()

        def e2e_step():
            # public host-buffer API: pinned input -> chunk-pipelined H2D / kernels / D2H -> pinned outputs
            vq.forward_host(x_host, n_chunks=E2E_CHUNKS, out=(q_host, i_host, l_host))

        for _ in range(max(3, min(args.warmup, 5))):   # >= 3: every chunk's pointer set is seen twice before it replays
            e2e_step()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            e2e_step()
        f1.record()
        barrier()
        ms_e2e = max_over_ranks(f0.elapsed_time(f1) / args.steps)
        h2d = x_host.numel() * x_host.element_size()
        d2h = q_host.numel() * 2 + i_host.numel() * 8 + 4
        e2e = {"value": world * n_vec / (ms_e2e * 1e-3), "unit": "vectors/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "numa_pinning": numa}
    elif os.environ.get("VQB_BENCH_SKIP_E2E"):  # profiling aid: keep the launch list to the device-resident steps
        if rank == 0:
            print(json.dumps({"ms_per_step": ms_dev, "kernel_ms": assign_ms, "gpu_launches": launches, "host_ms_per_step": host_ms}))
        if world > 1:
            dist.destroy_process_group()
        return

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = load_peaks()
    stages = 16 if cfg5 else 1
    d_stage = D // 2 if cfg5 else D
    flops = 2.0 * n_vec * K * d_stage  # algorithmic, per search launch: one pass of the N x K x D contraction (SURVEY 8d)
    # The kernel was timed alone between two events inside a step of a few-millisecond region at boost clocks: the
    # BURST peak is the honest denominator (B200_PROFILING.md); the sustained block carries its own fraction.
    peak_tf = peaks["bf16_tflops"]
    ach = flops / (assign_ms * 1e-3) / 1e12 if assign_ms else None
    roof = {"bound": "tensor", "kernel": "vq_assign_kernel (tcgen05 distance MMA + fused arg-max)",
            "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf if ach else None,
            "peak_source": peak_src + " bf16_tflops (burst: kernel event-timed inside a short region at boost clocks)",
            "kernel_ms": assign_ms, "kernel_share_of_step": assign_ms * stages / ms_dev_events if assign_ms else None,
            "measured": "CUDA event pair on the launching stream around every vq_assign_kernel launch, over the same K "
                        "steps repeated right after the headline region (events split the step's CUDA graph)",
            "ms_per_step_with_events": ms_dev_events,
            "algorithmic_flops_per_launch": flops, "executed_mma_passes": 3 if cfg5 else 2, "traffic": ncu_dram_bytes(),
            "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum of the launch AS BENCHED, fused tail on; "
                            "profiles/r2_assign_benched_summary.txt)"}
    if sustained and sustained["kernel_ms"]:
        pk = peaks.get("bf16_tflops_sustained", peak_tf)
        sustained["kernel_tflops"] = flops / (sustained["kernel_ms"] * 1e-3) / 1e12
        sustained["frac_of_sustained_peak"] = sustained["kernel_tflops"] / pk
        sustained["peak"] = pk
        sustained["peak_source"] = peak_src + " bf16_tflops_sustained"
    cpu_v = time_cpu(steps=2, warmup=1)[0] if world == 1 else None   # reported baseline: rank 0 at N=1 only
    line = {
        "metric": METRIC, "value": world * n_vec / (ms_dev * 1e-3), "unit": "vectors/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": "strong" if cfg5 else "weak",
        "vs_baseline": None, "dtype": "f32" if cfg5 else "bf16", "data": "synthetic",
        "config": {"workload": workload, "per_gpu_vectors": n_vec, "global_vectors": world * n_vec,
                   "parallelism": f"dp{world}: batch sharded, packed EMA statistics summed over the ranks once per step" if world > 1 else "single GPU",
                   "l2": "input (134 MB) + output (134 MB) per step exceed the 126 MB L2; no extra flush",
                   "index_mismatch_policy": "bit-exact vs the reference fixtures outside fp32 near-ties (tests/test_big_golden.py)"},
        "e2e": e2e,
        "gpu_launches": launches,
        "host_ms_per_step": host_ms,
        "clocks": clocks,
        "roofline": roof,
        "sustained": sustained,
        "cpu_baseline": cpu_baseline_block(cpu_v) if cpu_v is not None else None,
    }
    if cfg5:
        line["stage_vectors_per_s"] = world * n_vec * 16 / (ms_dev * 1e-3)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg5"],
                    help="cfg2 = BASELINE.json configs[1] (the headline, default); cfg5 = configs[4], GroupedResidualVQ, strong scaling")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 2 s sustained-clock block")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR as .npy files")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
