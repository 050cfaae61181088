#!/usr/bin/env python
"""bench.py -- binaural audio frames/s (RIR conv + spectrogram) on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm

A "step" is one pass of the hot path over one batch of synthetic input: every
env's 1-s source clip is convolved with its binaural RIR and turned into the
(65, T', 2) log-magnitude spectrogram (reference: soundspaces/simulator.py:608-701
+ soundspaces/tasks/nav.py:86-100).  Workload = BASELINE.json configs[1]: 128 envs
per GPU, 44.1 kHz, 16384-tap RIRs, output (128, 65, 69, 2); weak scaling (each
rank renders its own 128 envs; no data-path collective, as in the reference's
DD-PPO where observations never cross ranks).

Prints ONE JSON line on rank 0 (see the field notes in DESIGN.md section "Measurement").
"""
from __future__ import annotations

import argparse
import json
import os

# worker processes of the CPU arm are single-threaded (one env per process, like the reference's
# VectorEnv workers): must be set before numpy/scipy are imported in the spawned children
for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_k, "1")
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the modules imported from the tree leave nothing in it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "binaural audio frames/sec (RIR conv+STFT)"
UNIT = "frames/s"

# workload (BASELINE.json configs[1]; SURVEY.md 8(d) C2)
SR = 44100
TAPS = 16384
ENVS_PER_GPU = 128
N_BANKS = 16            # RIR banks rotated between steps: 16 x 16.8 MB = 268 MB > 126 MB L2
# SURVEY.md 8(d): bytes = 8*L_eff + 4*S/B_share + 8*65*T'  (spectrogram-only output)
ALG_BYTES_PER_FRAME = 8 * TAPS + 4 * SR // ENVS_PER_GPU + 8 * 65 * 69
# dram__bytes_read.sum + dram__bytes_write.sum per 64-env launch from the committed capture
# profiles/prof_r01d.ncu-rep (ncu --set full, cold-cache replay), by kernel
NCU_DRAM_BYTES_PER_LAUNCH = {"fwd_rir_kernel": 8.42e6, "mac_bins_kernel": 17.79e6, "mac_ifft_kernel": 46.86e6,
                             "spectrogram_kernel": 22.62e6}
# same capture: FMA-pipe busy cycles per SM (sm__pipe_fma_cycles_active.avg) and executed warp-instructions
# (smsp__inst_executed.sum) of one 64-env launch of each kernel -- the compute roofline this FP32 path really has
NCU_FMA_PIPE_CYCLES_PER_LAUNCH = {"fwd_rir_kernel": 4663.0, "mac_bins_kernel": 8912.0, "mac_ifft_kernel": 13389.0,
                                  "spectrogram_kernel": 21105.0}
NCU_WARP_INST_PER_LAUNCH = {"fwd_rir_kernel": 2.359e6, "mac_bins_kernel": 5.456e6, "mac_ifft_kernel": 8.000e6,
                            "spectrogram_kernel": 11.864e6}
ALG_FLOP_PER_FRAME = 17.3e6   # SURVEY.md 8(d): 2 packed 65536-pt FFT equivalents + mul + 276 packed 512-pt FFTs
FP32_PEAK_TFLOPS = 75.0       # nominal B200 FP32 SIMT, SURVEY.md 8(d)


def workload_config(n_gpus):
    return {
        "workload": "C2: 128 envs/GPU x (1-s 44.1 kHz source (*) 16384-tap binaural RIR -> (65,69,2) log-spectrogram)",
        "sr": SR, "rir_taps": TAPS, "envs_per_gpu": ENVS_PER_GPU, "global_envs": ENVS_PER_GPU * n_gpus,
        "spectrogram": [65, 69, 2], "stft_pad_mode": "reflect", "source": "one shared clip per batch",
        "l2_policy": f"inputs larger than L2: {N_BANKS} RIR banks ({N_BANKS * ENVS_PER_GPU * TAPS * 8 / 1e6:.0f} MB) rotated per step",
        "parallelism": f"env-sharded x{n_gpus}, no data-path collective",
    }


def make_bank_host(n_envs, seed0=0):
    """(n_envs, TAPS, 2) float32: N(0,1)*exp(-t/tau), tau = L/6, max|rir| = 0.5 (SURVEY.md 8(d));
    2 % of envs get the zero-RIR fallback."""
    rng = np.random.default_rng(1234 + seed0)
    env = np.exp(-np.arange(TAPS) / (TAPS / 6.0)).astype(np.float32)
    out = np.empty((n_envs, TAPS, 2), dtype=np.float32)
    for i in range(n_envs):
        r = rng.standard_normal((TAPS, 2), dtype=np.float32) * env[:, None]
        r *= np.float32(0.5) / np.abs(r).max()
        out[i] = r
    out[rng.random(n_envs) < 0.02] = 0.0
    return out


def silent_mask(n_envs, seed0=0):
    return np.random.default_rng(99 + seed0).random(n_envs) < 0.05      # 5 % silent envs


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.samples = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [l for (t, l) in self.samples if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.samples]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in rows:
            p = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except Exception:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU arm
def usable_cpus():
    """Host threads this process may really use: min(sched affinity, cgroup CPU quota)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:                                     # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:                                 # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def _cpu_init():
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"


def _cpu_frames(args):
    """Worker: render `count` frames of the C2 workload with the oracle (the reference's algorithm:
    scipy.signal.fftconvolve x2 ears + librosa.stft restatement + 4x4 mean + log1p)."""
    seed, count = args
    from oracle import audio_oracle as ao
    from synth import make_rir, make_source
    src = make_source(7, SR)
    rirs = [make_rir(seed * 4 + j, TAPS) for j in range(4)]
    t0 = time.perf_counter()
    acc = 0.0
    for i in range(count):
        _, spec = ao.render_frame(src, rirs[i % 4], SR)
        acc += float(spec[0, 0, 0])
    return time.perf_counter() - t0, acc


def cpu_throughput(frames_total, procs):
    """frames/s of the oracle on `procs` host processes (one env per task, single-threaded BLAS/FFT
    per process -- the reference's process-per-env model, ss_baselines/common/env_utils.py:41-106)."""
    import multiprocessing as mp
    per = max(1, frames_total // procs)
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs, initializer=_cpu_init) as pool:
        pool.map(_cpu_frames, [(i, 2) for i in range(procs)])          # warm-up / import
        t0 = time.perf_counter()
        pool.map(_cpu_frames, [(i, per) for i in range(procs)])
        dt = time.perf_counter() - t0
    return per * procs / dt, per * procs, dt


def run_reference(args, rank):
    """--impl reference: the reference's own CPU algorithm for the path, all host threads."""
    if rank != 0:
        return
    cores = usable_cpus()
    per_step = max(cores * 32, 64)       # bounded sample per step (about 0.15 s of wall time on 16 cores)
    vals = []
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    per = max(1, per_step // cores)
    with ctx.Pool(cores, initializer=_cpu_init) as pool:
        for _ in range(max(1, min(args.warmup, 2))):
            pool.map(_cpu_frames, [(i, per) for i in range(cores)])
        t0 = time.perf_counter()
        steps = args.steps
        for _ in range(steps):
            pool.map(_cpu_frames, [(i, per) for i in range(cores)])
        dt = time.perf_counter() - t0
    value = steps * per * cores / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 2), "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} steps x {per * cores} frames of the C2 workload, {cores} processes x 1 thread "
                                   "(oracle/audio_oracle.py: scipy.signal.fftconvolve + restated librosa.stft/block_reduce)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
def timed_region(step, steps, barrier, torch, first_index=0):
    """CUDA-event time in ms of exactly `steps` calls of step(i), barrier + synchronize on both sides: --steps is the
    number of steps every timed region runs, whatever its length."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e1.record()                     # an event is created by its first record: keep that out of the timed window
    barrier()
    e0.record()
    for i in range(steps):
        step(first_index + i)
    e1.record()
    barrier()
    return e0.elapsed_time(e1)


def numa_bind(local_rank, torch):
    """Bind this rank (and therefore the pinned buffers it allocates afterwards, first touch) to the CPUs of the
    NUMA node its GPU hangs off: eight unpinned ranks pushing 16 MB per step through one socket's memory is what held
    the round-1 end-to-end scaling at 0.67 (VERDICT r1).  Best effort: returns a description or the reason it did nothing."""
    try:
        from soundspaces_b200.distributed import gpu_numa_cpus
        node, cpus = gpu_numa_cpus(local_rank)
        if node is None or not cpus:
            return "no NUMA information for this GPU"
        allowed = os.sched_getaffinity(0)
        use = sorted(set(cpus) & set(allowed))
        if not use:
            return f"NUMA node {node}: none of its CPUs is in this process's cpuset"
        os.sched_setaffinity(0, use)
        return f"rank bound to NUMA node {node} ({len(use)} CPUs)"
    except Exception as e:          # noqa: BLE001
        return "not bound: " + repr(e)[:80]


# LIVE figures of one step of the C2 workload, per convolution plan, from the committed range captures (scratch/prof_final.sh:
# `ncu --replay-mode range --cache-control none` around 4 consecutive steady-state steps, both internal streams running
# concurrently, caches as the previous steps left them): DRAM / L2 bytes and the time the FMA pipes / issue slots were busy
LIVE_STEP = os.path.join(ROOT, "profiles", "live_step_r02b.json")
# FMA-pipe cycles per SM and executed warp-instructions per launch from the committed `ncu --set full` captures, by kernel
# (64-env launches of the C2 workload): the per-kernel view of the same thing
NCU_PER_LAUNCH = os.path.join(ROOT, "profiles", "ncu_per_launch.json")


def read_live_step(path_name):
    try:
        d = json.load(open(LIVE_STEP))[path_name]
        return {"dram_bytes": d["dram_bytes_per_step"], "l2_bytes": d["l2_bytes_per_step"], "fma_busy_us": d["fma_pipe_busy_us_per_step"],
                "issue_busy_us": d["issue_busy_us_per_step"], "source": d["source"]}
    except Exception:
        return None


def alg_bytes(taps_eff, src_samples, share, sr):
    """SURVEY.md 8(d): 8*L_eff + 4*S_seg/B_share + 8*65*T' (spectrogram-only output)."""
    cols = -(-(1 + sr // 160) // 4)
    return 8 * taps_eff + 4 * src_samples // max(share, 1) + 8 * 65 * cols


def run_gpu(args, rank, local_rank, world):
    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL prints its version there)
    # are sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    numa = numa_bind(local_rank, torch) if (world > 1 and not args.no_numa) else "single rank: not bound"
    import torch.distributed as dist
    from soundspaces_b200 import AudioRequest, BatchedAudioRenderer
    from synth import make_rir, make_source

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        # a collective that some rank never reaches must not hang the box: abort after 3 minutes
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))

    B = ENVS_PER_GPU
    r = BatchedAudioRenderer(SR, TAPS, device=dev, log2n=args.log2n, prefer_block64=(args.plan == "block64"))
    r.set_conv_mode(args.conv_mode)
    sid = r.add_source(make_source(7, SR))
    bank_host = make_bank_host(N_BANKS * B, seed0=rank)
    bank = torch.from_numpy(bank_host).to(dev)
    ids = r.set_dense_rir_bank(bank)
    sil = silent_mask(B, seed0=rank)
    req_lists = [[AudioRequest(rir=ids[k * B + i], source=sid, silent=bool(sil[i])) for i in range(B)] for k in range(N_BANKS)]
    batches = [r.prepare(q) for q in req_lists]
    path = "block64" if batches[0].plan.log2n == 16 else "partitioned"
    spec_out = torch.empty((B,) + r.spec_shape, dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def agree(ok):
        """True only when EVERY rank succeeded.  The optional legs below set up rank-locally inside try / except and
        call this before their first collective, so that a rank that failed (out of pinned memory, ...) cannot leave
        the others waiting in a barrier."""
        if world == 1:
            return bool(ok)
        t = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item() == 1.0)

    def step(i):
        r.execute(batches[i % N_BANKS], out=spec_out)

    # ---- device-resident throughput ("value")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    for i in range(args.warmup):
        step(i)
    barrier()
    launches0 = r.ctx.launch_count
    t_wall0 = time.time()
    ms = timed_region(step, args.steps, barrier, torch)
    t_wall1 = time.time()
    launches = r.ctx.launch_count - launches0
    if args.dump_outputs:
        # what the caller of the timed path received from its last step: the spectrogram batch of that step
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "spectrogram" if world == 1 else f"spectrogram_rank{rank}"
        np.save(os.path.join(args.dump_outputs, name + ".npy"), spec_out.cpu().numpy())
    # a long enough region for the clock sampler: keep the GPU under the same load for >= 1.5 s
    clocks = None
    if sampler:
        t_end = time.time() + max(0.0, 1.5 - (t_wall1 - t_wall0))
        i = 0
        while time.time() < t_end:
            for _ in range(50):
                step(i); i += 1
            torch.cuda.synchronize()
        t_wall1 = time.time()
        clocks = sampler.stop(t_wall0, t_wall1)
    ms_max = allmax(ms)

    # ---- centralised-policy mode (SURVEY.md 8(e)): every step ends with ONE in-place all-gather of the observation
    # batch; the spectrogram kernel writes straight into this rank's slice of the gather buffer
    gather_info = None
    if world > 1 and not args.no_gather:
        err = None
        try:
            from soundspaces_b200.distributed import GatheredObservations
            gobs = GatheredObservations(B * world, r.spec_shape, rank, world, dev)
            assert gobs.n_local == B
            state = {}

            def gstep(i):
                r.execute(batches[i % N_BANKS], out=gobs.local)
                state["flat"] = gobs.gather()
        except Exception as e:          # noqa: BLE001
            err = repr(e)[:200]
        if not agree(err is None):
            gather_info = {"error": err or "set-up failed on another rank"}
    if world > 1 and not args.no_gather and gather_info is None:
        try:
            for i in range(max(3, args.warmup // 2)):
                gstep(i)
            gms = timed_region(gstep, args.steps, barrier, torch)
            gms = allmax(gms)
            # every rank must now hold every rank's rows: compare a checksum of the gathered batch across ranks,
            # and this rank's own rows with what it rendered without the collective
            flat = state["flat"]
            chk = flat.double().sum().reshape(1)
            lo, hi = chk.clone(), chk.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            r.execute(batches[(args.steps - 1) % N_BANKS], out=spec_out)
            own = torch.tensor([float(torch.equal(gobs.local, spec_out))], device=dev)
            dist.all_reduce(own, op=dist.ReduceOp.MIN)
            gather_info = {"value": B * world * args.steps / (gms * 1e-3), "unit": UNIT,
                           "ms_per_step": gms / args.steps, "cost_ms_per_step": gms / args.steps - ms_max / args.steps,
                           "bytes_sent_per_rank_per_step": int(gobs.local.numel() * 4),
                           "collective": "one in-place ncclAllGather per step (all_gather_into_tensor on the buffer the "
                                         "spectrogram kernel wrote into)",
                           "identical_on_all_ranks": bool(float(lo.item()) == float(hi.item())),
                           "local_rows_bit_identical_to_ungathered": bool(own.item() == 1.0)}
        except Exception as e:          # informational leg: never take the headline measurement down with it
            gather_info = {"error": repr(e)[:200]}

    # ---- per-kernel durations for the roofline (same K steps, events around every launch)
    r.ctx.set_kernel_timing(True)
    for i in range(args.steps):
        step(i)
    ktimes = r.ctx.get_kernel_timing()
    r.ctx.set_kernel_timing(False)

    # ---- end to end through the host-buffer C-ABI entry ("e2e")
    hs = r.make_host_session(B, TAPS, want_wave=False, n_chunks=args.chunks)
    hs.h_rir.numpy()[:] = bank_host[:B]
    hs.set_requests(sid, silent=sil)
    for _ in range(max(3, args.warmup // 4)):
        hs.run()
    e2e_ms = timed_region(lambda i: hs.run(), args.steps, barrier, torch)
    e2e_ms_max = allmax(e2e_ms)
    checksum = float(hs.h_spec.double().sum())
    hs_bytes = (hs.h2d_bytes, hs.d2h_bytes)

    # ---- end to end with a device-resident RIR bank and a stated miss rate (SURVEY.md N1: what training does once the
    # scene's working set is resident: per step only the MISSING RIRs cross PCIe, the spectrograms come back)
    miss_info = None
    err = None
    try:
        miss = args.miss_rate
        n_miss = max(1, int(round(miss * B)))
        h_miss = torch.from_numpy(bank_host[:n_miss].copy()).pin_memory()
        d_miss = [torch.empty((n_miss, TAPS, 2), dtype=torch.float32, device=dev) for _ in range(2)]
        h_spec = [torch.empty((B,) + r.spec_shape, dtype=torch.float32).pin_memory() for _ in range(2)]
        d_spec = [torch.empty((B,) + r.spec_shape, dtype=torch.float32, device=dev) for _ in range(2)]
        copy_stream, back_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        ev = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]          # kernels of step i finished writing d_spec[i & 1]
        ev_back = [torch.cuda.Event() for _ in range(2)]          # D2H of d_spec[i & 1] finished
        state = {"n": 0}

        def mstep(i):
            k = state["n"] & 1
            state["n"] += 1
            main = torch.cuda.current_stream(dev)
            with torch.cuda.stream(copy_stream):                    # the misses of step i+1 travel during step i
                d_miss[k].copy_(h_miss, non_blocking=True)
                ev[k].record(copy_stream)
            main.wait_event(ev[k])
            # the uploaded rows replace the first n_miss rows of this step's bank slice (same request array)
            bank[(i % N_BANKS) * B: (i % N_BANKS) * B + n_miss].copy_(d_miss[k], non_blocking=True)
            main.wait_event(ev_back[k])                              # d_spec[k] was read back two steps ago
            r.execute(batches[i % N_BANKS], out=d_spec[k])
            ev_done[k].record(main)
            with torch.cuda.stream(back_stream):                    # the read-back overlaps the next step's kernels
                back_stream.wait_event(ev_done[k])
                h_spec[k].copy_(d_spec[k], non_blocking=True)
                ev_back[k].record(back_stream)

        def mbarrier():
            barrier()
            back_stream.synchronize()

        for i in range(6):
            mstep(i)
        torch.cuda.synchronize()
    except Exception as e:          # noqa: BLE001
        err = repr(e)[:200]
    if not agree(err is None):
        miss_info = {"error": err or "set-up failed on another rank"}
    try:
        if miss_info is not None:
            raise RuntimeError(miss_info["error"])
        mms = timed_region(mstep, args.steps, mbarrier, torch)
        mms = allmax(mms)
        miss_info = {"value": B * world * args.steps / (mms * 1e-3), "unit": UNIT, "ms_per_step": mms / args.steps,
                     "miss_rate": n_miss / B, "h2d_bytes_per_step": int(n_miss * TAPS * 8),
                     "d2h_bytes_per_step": int(h_spec[0].numel() * 4),
                     "what": "device-resident bank; per step the missing RIRs are copied from pinned host memory on a copy "
                             "stream and the spectrograms are read back on another (both overlap the neighbouring steps' kernels; the "
                             "timed region ends when the last read-back has landed)"}
        bank.copy_(torch.from_numpy(bank_host))                      # restore for the legs below
        torch.cuda.synchronize()
    except Exception as e:          # noqa: BLE001
        miss_info = {"error": repr(e)[:200]}

    # ---- the public API paths (VERDICT r1 weak #3/#4): per step host work included
    api_info = {}
    err = None
    try:
        def api_step(i):                                            # render(list[AudioRequest]): prepare() every step
            r.execute(r.prepare(req_lists[i % N_BANKS]), out=spec_out)
        for i in range(5):
            api_step(i)
        rir_arr = [np.asarray(ids[k * B:(k + 1) * B], dtype=np.int64) for k in range(N_BANKS)]

        def arr_step(i):                                            # prepare_arrays(): requests held as arrays
            r.execute(r.prepare_arrays(rir_arr[i % N_BANKS], sid, silent=sil), out=spec_out)
        for i in range(5):
            arr_step(i)
        torch.cuda.synchronize()
    except Exception as e:          # noqa: BLE001
        err = repr(e)[:200]
    ok_api = agree(err is None)
    try:
        if not ok_api:
            raise RuntimeError(err or "set-up failed on another rank")
        ams = timed_region(api_step, args.steps, barrier, torch)
        bms = timed_region(arr_step, args.steps, barrier, torch)
        api_info = {"api_path": {"value": B * world * args.steps / (allmax(ams) * 1e-3), "unit": UNIT,
                                 "what": "execute(prepare(list[AudioRequest])) every step: request resolution + H2D of the request array + launches"},
                    "api_path_arrays": {"value": B * world * args.steps / (allmax(bms) * 1e-3), "unit": UNIT,
                                        "what": "execute(prepare_arrays(...)) every step: requests held as numpy columns"}}
    except Exception as e:          # noqa: BLE001
        api_info = {"api_path": {"error": repr(e)[:200]}}
    api_info["plugin_path"] = plugin_path_leg(args, r, bank_host, sid, dev, world, barrier, allmax, agree, torch)

    # ---- the other convolution plan on the same workload (N = 1): the single-block cluster kernel trades step time
    # for DRAM traffic (no H / Y intermediates); reported next to the headline, which uses the faster plan
    alt = None
    if world == 1 and not args.no_extra:
        try:
            other = "partitioned" if path == "block64" else "block64"
            r2 = BatchedAudioRenderer(SR, TAPS, device=dev, prefer_block64=(other == "block64"))
            sid2 = r2.add_source(make_source(7, SR))
            ids2 = r2.set_dense_rir_bank(bank)
            b2 = [r2.prepare([AudioRequest(rir=ids2[k * B + i], source=sid2, silent=bool(sil[i])) for i in range(B)]) for k in range(N_BANKS)]
            out2 = torch.empty_like(spec_out)

            def step2(i):
                r2.execute(b2[i % N_BANKS], out=out2)
            for i in range(args.warmup):
                step2(i)
            ms2 = timed_region(step2, args.steps, barrier, torch)
            r2.ctx.set_kernel_timing(True)
            for i in range(args.steps):
                step2(i)
            kt2 = r2.ctx.get_kernel_timing()
            r2.ctx.set_kernel_timing(False)
            step(0); step2(0)
            torch.cuda.synchronize()
            live2 = read_live_step(other)
            alt = {"plan": other, "value": B * args.steps / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2 / args.steps,
                   "kernel_ms_all": {k: v[0] / args.steps for k, v in kt2.items() if v[1]},
                   "traffic": live2["dram_bytes"] if live2 else None, "traffic_source": live2["source"] if live2 else None,
                   "traffic_over_algorithmic": (live2["dram_bytes"] / (ALG_BYTES_PER_FRAME * B)) if live2 else None,
                   "fma_pipe_frac_live": (live2["fma_busy_us"] / (ms2 / args.steps * 1e3)) if live2 else None,
                   "max_abs_diff_vs_headline_plan": float((out2 - spec_out).abs().max())}
            del r2, b2
        except Exception as e:          # noqa: BLE001
            alt = {"error": repr(e)[:200]}

    extra = None
    if world == 1 and not args.no_extra:
        del hs
        extra = extra_workloads(args, dev, torch, barrier)

    if rank == 0:
        frames = B * world * args.steps
        value = frames / (ms_max * 1e-3)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
        else:
            peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
        hot = [k for k in ("fwd_rir_kernel", "mac_bins_kernel", "mac_ifft_kernel", "conv64k_kernel", "spectrogram_kernel") if ktimes[k][1]]
        # per STEP: a kernel may be launched several times per step (sub-batches on internal streams)
        per_step_ms = {k: ktimes[k][0] / args.steps for k in hot}
        launches_per_step = {k: ktimes[k][1] / args.steps for k in hot}
        dom = max(hot, key=lambda k: per_step_ms[k])
        dom_ms = per_step_ms[dom]
        alg_bytes_launch = ALG_BYTES_PER_FRAME * B            # all of the step's frames pass through every kernel
        achieved = alg_bytes_launch / (dom_ms * 1e-3) / 1e9
        step_ms = ms_max / args.steps
        kernel_sum = sum(per_step_ms.values())
        live = read_live_step(path)
        # compute roofline of the kernels as built: the time the FMA pipes / the issue slots need for one step's
        # instructions (counts per launch from the committed ncu capture) over the measured step time
        fma_frac = issue_frac = None
        try:
            per_launch = json.load(open(NCU_PER_LAUNCH))[path]
            sm_mhz = ((clocks or {}).get("sm_mhz") or 1965.0)
            sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
            fma_frac = (sum(per_launch[k]["fma_pipe_cycles_per_sm"] * launches_per_step[k] for k in hot)
                        / (sm_mhz * 1e6) / (step_ms * 1e-3))
            issue_frac = (sum(per_launch[k]["warp_instructions"] * launches_per_step[k] for k in hot)
                          / (sm_count * 4) / (sm_mhz * 1e6) / (step_ms * 1e-3))
        except Exception:
            pass
        cfg = workload_config(world)
        cfg["convolution_plan"] = ("single block: one fused 65536-point cluster kernel per env (conv64k_kernel)" if path == "block64"
                                   else "partitioned overlap-save (fwd_rir / mac_bins / mac_ifft)")
        cfg["numa"] = numa
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "timed_region_s": ms_max * 1e-3,
            "roofline": {
                "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": live["dram_bytes"] if live else None,
                "traffic_source": ("dram__bytes_read.sum + dram__bytes_write.sum per LIVE STEP of this workload (all kernels of the step; to be "
                                   "read against algorithmic_bytes_per_step): " + live["source"]) if live else None,
                "traffic_over_algorithmic": (live["dram_bytes"] / alg_bytes_launch) if live else None,
                "l2_bytes_per_step": live.get("l2_bytes") if live else None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_step": alg_bytes_launch, "kernel_ms": dom_ms,
                "kernel_ms_all": per_step_ms, "kernel_launches_per_step": launches_per_step,
                "kernel_timing": "CUDA events around every launch, summed per step; sub-batches run on 2 internal streams, "
                                 "so the per-kernel sums overlap in wall time",
                "kernel_share_of_step": dom_ms / max(kernel_sum, 1e-9),
                "path_achieved_gbs": alg_bytes_launch / (step_ms * 1e-3) / 1e9,
                "path_frac_hbm": alg_bytes_launch / (step_ms * 1e-3) / 1e9 / peak,
                "fp32_frac_nominal": (value / world) * ALG_FLOP_PER_FRAME / (FP32_PEAK_TFLOPS * 1e12),
                "fp32_lane_op_peak_measured": "36.6e12 FP32-pipe lane-ops/s (FADD2 / FFMA2 issue rate, profiles/f32x2_bench_r02.log): an "
                                              "add-dominated FFT can at most reach 36.6 TFLOP/s, not the 73 TFLOP/s of pure FMA code",
                "fma_pipe_frac": fma_frac, "issue_slot_frac": issue_frac,
                "fma_pipe_frac_live": (live["fma_busy_us"] / (step_ms * 1e3)) if live else None,
                "issue_slot_frac_live": (live["issue_busy_us"] / (step_ms * 1e3)) if live else None,
                "fma_pipe_note": "fma_pipe_frac: per-launch FMA-pipe cycles of the committed per-kernel captures x launches per step / this run's step time; "
                                 "fma_pipe_frac_live: FMA-pipe busy time per step measured over a live range of 4 steps / this run's step time",
                "note": "FFT work is FP32-pipe bound (about 100 flop/B at algorithmic traffic): fma_pipe_frac / issue_slot_frac are the "
                        "fractions that measure kernel quality; see DESIGN.md",
            },
            "e2e": {"value": B * world * args.steps / (e2e_ms_max * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": hs_bytes[0], "d2h_bytes_per_step": hs_bytes[1],
                    "ms_per_step": e2e_ms_max / args.steps, "api": f"ssb_render_batch_host (pinned host RIRs in, host spectrograms out), {args.chunks} pipelined chunks",
                    "checksum": checksum},
            "e2e_resident_bank": miss_info,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        line.update(api_info)
        if gather_info is not None:
            line["with_allgather"] = gather_info
        if alt is not None:
            line["alternative_plan"] = alt
        if extra is not None:
            line["extra_workloads"] = extra
        if world == 1 and not args.no_cpu:
            cores = usable_cpus()
            v, n, dt = cpu_throughput(cores * args.cpu_frames_per_core, cores)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{n} frames of the same C2 workload in {dt:.1f} s, {cores} processes x 1 thread "
                                              "(oracle/audio_oracle.py: scipy.signal.fftconvolve + restated librosa.stft/block_reduce)"}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def plugin_path_leg(args, r, bank_host, sid, dev, world, barrier, allmax, agree, torch):
    """Frames/s through the per-env plugin surface: SpectrogramSensor.get_observation per env (deferred handles) +
    batch_obs, every env at a NEW grid node every step (100 % memo miss, resident RIRs)."""
    err = None
    try:
        pstep = _plugin_setup(args, r, bank_host, sid, dev, torch)
        for i in range(5):
            pstep(i)
        torch.cuda.synchronize()
    except Exception as e:          # noqa: BLE001
        err = repr(e)[:200]
    if not agree(err is None):
        return {"error": err or "set-up failed on another rank"}
    B = ENVS_PER_GPU
    pms = timed_region(pstep, args.steps, barrier, torch)
    pms = allmax(pms)
    return {"value": B * world * args.steps / (pms * 1e-3), "unit": UNIT, "ms_per_step": pms / args.steps,
            "what": "per env: SpectrogramSensor.get_observation -> DeferredObservation handle; per step: batch_obs -> ONE render into "
                    "the rollout slot (128 envs, every env at a new node each step, RIRs resident)"}


def _plugin_setup(args, r, bank_host, sid, dev, torch):
    from soundspaces_b200.replay import ReplayScene, ReplaySim, ReplayVectorEnv
    from soundspaces_b200.sensors import batch_obs
    from soundspaces_b200.simulator import AudioRenderService
    from synth import make_source
    B = ENVS_PER_GPU
    svc = AudioRenderService(SR, device=dev, renderer=r)
    scene = ReplayScene("bench", side=46)                            # 2116 nodes >= 16 * 128 distinct positions
    n_rows = bank_host.shape[0]
    for recv in range(n_rows):                                       # the resident bank rows ARE the scene's RIRs (azimuth 0)
        svc._rir_ids[(scene.rir_dir, 0, recv, 0)] = recv
    clip = make_source(7, SR)
    svc._src_ids[("telephone", len(clip), id(clip))] = (sid, clip)
    sims = [ReplaySim(svc, scene, "telephone", clip, source_node=0, start_node=i) for i in range(B)]
    for s in sims:
        s.b200_prefetch = False
    envs = ReplayVectorEnv(sims)
    out = {"spectrogram": torch.empty((B,) + r.spec_shape, dtype=torch.float32, device=dev)}

    def pstep(i):
        base = (i % N_BANKS) * B
        for k, s in enumerate(sims):                                 # teleport: every env observes a new node (memo miss)
            s._receiver_position_index = base + k
            s._spectrogram_cache = {}
        batch_obs(envs.observe(), device=dev, out=out)

    return pstep


def extra_workloads(args, dev, torch, barrier):
    """The other BASELINE.json configs on ONE GPU, inputs resident (same timing rules, --steps steps each):
    C3 head / valid / log-mel at 512 envs, C4 (ambisonic decode + convolution) at 256 envs, C5 rollout (16 envs)."""
    from soundspaces_b200 import AudioRequest, BatchedAudioRenderer
    from synth import make_source
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    res = {}
    steps, warm = args.steps, 5
    rng = np.random.default_rng(0)
    sr, L, Bc = 16000, 48000, 512

    def run(name, fn, frames_per_step, bytes_per_frame, flop_per_frame, note):
        for i in range(warm):
            fn(i)
        ms = timed_region(fn, steps, barrier, torch)
        v = frames_per_step * steps / (ms * 1e-3)
        res[name] = {"value": v, "unit": UNIT, "ms_per_step": ms / steps, "envs": frames_per_step,
                     "algorithmic_bytes_per_frame": bytes_per_frame, "path_frac_hbm": v * bytes_per_frame / 1e9 / peak,
                     "algorithmic_flop_per_frame": flop_per_frame, "fp32_frac_nominal": v * flop_per_frame / (FP32_PEAK_TFLOPS * 1e12),
                     "workload": note}
    try:
        r = BatchedAudioRenderer(sr, L, device=dev)
        env = np.exp(-np.arange(L) / (L / 6.0)).astype(np.float32)
        banks = [torch.from_numpy((rng.standard_normal((Bc, L, 2)).astype(np.float32) * env[None, :, None] * 0.1)).to(dev) for _ in range(2)]
        bank = torch.cat(banks)                                          # 2 x 196 MB rotated: larger than L2
        ids = r.set_dense_rir_bank(bank)
        s1, s4 = r.add_source(make_source(1, sr)), r.add_source(make_source(2, 4 * sr))
        out = torch.empty((Bc,) + r.spec_shape, device=dev)
        head = [r.prepare([AudioRequest(rir=ids[k * Bc + i], source=s1) for i in range(Bc)]) for k in range(2)]
        valid = [r.prepare([AudioRequest(rir=ids[k * Bc + i], source=s4, offset=3 * sr) for i in range(Bc)]) for k in range(2)]
        plan = "single-block cluster kernel" if head[0].plan.log2n == 16 else "partitioned"
        run("C3_head", lambda i: r.execute(head[i & 1], out=out), Bc, alg_bytes(16000, 16000, 64, sr), 7.4e6,
            f"512 envs, 16 kHz, 1-s clip x 48000-tap RIRs (first 16000 taps matter) -> (65,26,2); {plan}")
        run("C3_valid", lambda i: r.execute(valid[i & 1], out=out), Bc, alg_bytes(48000, 63999, 64, sr), 13.2e6,
            f"512 envs, 16 kHz, 4-s clip steady state: all 48000 taps (mode='valid') -> (65,26,2); {plan}")
        mel_out = torch.empty((Bc,) + r.logmel_shape(64), device=dev)

        def logmel(i):
            r.logmel(r.convolve_prepared(valid[i & 1]), 64, 2, out=mel_out)
        run("C3_valid_logmel", logmel, Bc, 8 * 48000 + 4 * 63999 // 64 + 8 * 64 * 101, 13.2e6 + 101 * 2 * 2 * 2 * 257,
            f"as C3_valid with the log-mel head (64 Slaney mels, power 2; extension, parity unpinned) -> (64,101,2); {plan}")
        # the same two workloads on the single-block plan (48000 taps <= 65536 - 16000 + 1: one 65536-point kernel per env)
        r64 = BatchedAudioRenderer(sr, L, device=dev, prefer_block64=True)
        ids64 = r64.set_dense_rir_bank(bank)
        t1, t4 = r64.add_source(make_source(1, sr)), r64.add_source(make_source(2, 4 * sr))
        head64 = [r64.prepare([AudioRequest(rir=ids64[k * Bc + i], source=t1) for i in range(Bc)]) for k in range(2)]
        valid64 = [r64.prepare([AudioRequest(rir=ids64[k * Bc + i], source=t4, offset=3 * sr) for i in range(Bc)]) for k in range(2)]
        if head64[0].plan.log2n == 16:
            run("C3_head_block64", lambda i: r64.execute(head64[i & 1], out=out), Bc, alg_bytes(16000, 16000, 64, sr), 7.4e6,
                "C3_head on the single-block cluster kernel")
            run("C3_valid_block64", lambda i: r64.execute(valid64[i & 1], out=out), Bc, alg_bytes(48000, 63999, 64, sr), 13.2e6,
                "C3_valid on the single-block cluster kernel")
        del r, r64, bank, banks
    except Exception as e:          # noqa: BLE001
        res["C3_error"] = repr(e)[:200]
    try:
        B4 = 256
        r = BatchedAudioRenderer(sr, L, device=dev)
        amb = torch.randn((B4, L, 9), device=dev) * 0.05
        az = torch.tensor([0., 90., 180., 270.] * (B4 // 4))
        s4 = r.add_source(make_source(2, 4 * sr))
        out = torch.empty((B4,) + r.spec_shape, device=dev)
        rirs = r.sh_decode(amb, az)
        ids = r.set_dense_rir_bank(rirs)
        batch = r.prepare([AudioRequest(rir=i, source=s4, offset=3 * sr) for i in ids])

        def c4(i):
            r.set_dense_rir_bank(r.sh_decode(amb, az))
            r.execute(batch, out=out)
        run("C4_decode_conv", c4, B4, 36 * L + 8 * 65 * 26, 44e6,
            "256 envs: 9-channel ambisonic RIR (48000 taps) -> SH rotate + HRTF decode -> valid-mode convolution -> (65,26,2)")
        del r, amb
    except Exception as e:          # noqa: BLE001
        res["C4_error"] = repr(e)[:200]
    try:
        res["C1_single_env"] = c1_single_env(dev, torch, reps=args.steps)
    except Exception as e:          # noqa: BLE001
        res["C1_error"] = repr(e)[:200]
    try:
        res["C5_rollout"] = c5_rollout(dev, torch, num_steps=args.steps)
    except Exception as e:          # noqa: BLE001
        res["C5_error"] = repr(e)[:200]
    return res


def c1_single_env(dev, torch, reps, sr=44100, taps=22050):
    """BASELINE.json configs[0] (SURVEY C1): ONE env, 1-s clip at 44.1 kHz x 22050-tap binaural RIR read from a wav file on
    disk, through the reference's own per-env call: sim.get_current_spectrogram_observation(compute_spectrogram) -> host
    ndarray (compat mode: one render + blocking read-back per call; memo defeated by alternating two receiver nodes whose
    dict entries are dropped).  Latency per call next to the CPU port's time for the same frame on one core."""
    import tempfile
    from scipy.io import wavfile
    from soundspaces_b200.replay import ReplayScene, ReplaySim
    from soundspaces_b200.sensors import SpectrogramSensor
    from soundspaces_b200.simulator import AudioRenderService
    from oracle import audio_oracle as ao
    from synth import make_rir, make_source
    svc = AudioRenderService(sr, device=dev, max_taps=sr, n_terms=1)
    clip = make_source(3, sr)
    with tempfile.TemporaryDirectory() as d:
        scene = ReplayScene("apartment_0", side=2, rir_root=d)
        rirs = [make_rir(900 + i, taps) for i in range(2)]
        for i in range(2):
            os.makedirs(os.path.join(scene.rir_dir, "0"), exist_ok=True)
            wavfile.write(os.path.join(scene.rir_dir, "0", f"{i}_3.wav"), sr, rirs[i])
        sim = ReplaySim(svc, scene, "telephone.wav", clip, source_node=3, start_node=0, deferred=False)
        sim.b200_prefetch = False
        fn = SpectrogramSensor.compute_spectrogram
        first = time.perf_counter()
        spec = sim.get_current_spectrogram_observation(fn)              # cold: wav read + upload + source spectrum
        cold_ms = (time.perf_counter() - first) * 1e3
        t0 = time.perf_counter()
        for i in range(reps):
            sim._receiver_position_index = i & 1
            sim._spectrogram_cache, sim._audiogoal_cache = {}, {}
            spec = sim.get_current_spectrogram_observation(fn)
        gpu_ms = (time.perf_counter() - t0) * 1e3 / reps
        t0 = time.perf_counter()
        for i in range(5):
            _, ref = ao.render_frame(clip, rirs[i & 1], sr)
        cpu_ms = (time.perf_counter() - t0) * 1e3 / 5
        ok = bool(np.allclose(spec, ao.render_frame(clip, rirs[(reps - 1) & 1], sr)[1], rtol=1e-4, atol=1e-5))
    return {"value": 1e3 / gpu_ms, "unit": UNIT, "ms_per_call": gpu_ms, "first_call_ms": cold_ms, "cpu_port_ms_per_frame_one_core": cpu_ms,
            "matches_oracle": ok,
            "workload": "1 env, 44.1 kHz, 22050-tap RIR from a wav file, compat path: get_current_spectrogram_observation -> host ndarray "
                        "(render B=1 + blocking device->host copy per call; RIR resident after the first read)"}


def c5_rollout(dev, torch, num_steps, n_envs=16, sr=16000, taps=16000):
    """BASELINE.json configs[4]: DD-PPO rollout, 16 envs per GPU, audio observation fused into the step (trace-replay
    env, SURVEY.md 8(d)): env-steps/s with the env_time / pth_time split of ppo_trainer.py:125-194."""
    from soundspaces_b200.replay import AudioPolicy, ReplayScene, ReplaySim, ReplayVectorEnv, collect_rollout
    from soundspaces_b200.simulator import AudioRenderService
    from synth import make_rir, make_source
    svc = AudioRenderService(sr, device=dev, max_taps=taps, n_terms=1)
    scene = ReplayScene("apartment_replay", side=8)
    rng = np.random.default_rng(11)
    base = np.stack([make_rir(500 + i, taps) for i in range(8)])
    mix = rng.standard_normal((4, scene.n_nodes, 8)).astype(np.float32) / 3.0
    rirs = np.einsum("anb,ble->anle", mix, base).astype(np.float32)          # [azimuth][node](taps, 2)
    scene.register_rirs(svc, source=0, rirs=rirs)
    clip = make_source(21, sr)
    sims = [ReplaySim(svc, scene, "telephone.wav", clip, source_node=0, start_node=int(rng.integers(scene.n_nodes)),
                      start_rotation=int(rng.integers(4)) * 90) for _ in range(n_envs)]
    envs = ReplayVectorEnv(sims)
    policy = AudioPolicy(svc.renderer.spec_shape).to(dev)
    storage = torch.zeros((num_steps + 1, n_envs) + svc.renderer.spec_shape, device=dev)
    trace = rng.choice([1, 1, 1, 2, 3], size=(num_steps, n_envs))              # recorded action trace (no STOP)
    collect_rollout(envs, policy, storage, min(20, num_steps), trace[:min(20, num_steps)])   # warm-up
    l0, f0 = svc.renderer.ctx.launch_count, svc.batcher.flushes
    t0 = time.time()
    pth, env_t, n = collect_rollout(envs, policy, storage, num_steps, trace, fused=True)
    wall = time.time() - t0
    rendered = sum(len(s._spectrogram_cache) for s in sims)
    return {"value": n / wall, "unit": "env-steps/s", "envs": n_envs, "num_steps": num_steps, "env_time_s": env_t, "pth_time_s": pth,
            "wall_s": wall, "renders": svc.batcher.flushes - f0, "kernel_launches": svc.renderer.ctx.launch_count - l0,
            "memo_entries": rendered, "rir_miss_rate": svc.miss_rate,
            "workload": "trace-replay env (8x8 grid scene, 16 kHz, 16000-tap RIRs resident) x SpectrogramSensor (deferred) x batch_obs into "
                        "rollouts.observations['spectrogram'][step+1] x AudioCNN-shaped policy (first layer: the fused permute + Conv2d + ReLU "
                        "kernel, SURVEY N2); ONE render per step for all envs"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2n", type=int, default=0)
    ap.add_argument("--conv-mode", type=int, default=0, help="0: mac_bins + ifft kernels, 1: fused mac_ifft")
    ap.add_argument("--plan", default="partitioned", choices=["partitioned", "block64"],
                    help="convolution plan of the headline leg: partitioned overlap-save (fastest) or the single-block cluster kernel (least traffic)")
    ap.add_argument("--chunks", type=int, default=2, help="pipeline depth of the host-buffer (e2e) entry")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--gather", action="store_true", help="(default for N > 1; kept for old command lines)")
    ap.add_argument("--no-gather", action="store_true",
                    help="N > 1: skip the centralised-policy leg (one in-place all-gather of the observations per step)")
    ap.add_argument("--cpu-frames-per-core", type=int, default=150)
    ap.add_argument("--no-extra", action="store_true", help="N = 1: skip the other BASELINE configs (extra_workloads)")
    ap.add_argument("--no-numa", action="store_true", help="N > 1: do not bind ranks to their GPU's NUMA node")
    ap.add_argument("--miss-rate", type=float, default=0.10, help="e2e_resident_bank: fraction of envs whose RIR is uploaded per step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the spectrogram batch the timed path returned in its last step to DIR/spectrogram.npy "
                         "(float32; one file per rank, spectrogram_rank<r>.npy, when --gpus > 1)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            # convenience: re-launch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29511"),
                   os.path.abspath(__file__)] + sys.argv[1:]
            sys.exit(subprocess.call(cmd))
        raise SystemExit(f"WORLD_SIZE={world} does not match --gpus {args.gpus}")
    run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
