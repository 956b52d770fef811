#!/usr/bin/env python
"""bench.py -- headline benchmark: voice-samples/s of the 65 536-voice
SineGen -> Lopass(SVF) -> gain chain at 48 kHz (BASELINE.json metric, SURVEY.md 8d "Config A").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own SSE path on host cores

One "step" = one pass of the hot path over one batch: T = 64 blocks (4096 samples, 85 ms of
audio) for every voice = ONE fused kernel launch (contract R: per-voice signal-rate frequency
rows in, per-voice output rows out, reference layout [T][V][64] f32) plus the mix-bus
partial sums and their tiny reduce kernel.  Inputs are resident in HBM before the timed
region; in + out = 2.1 GB per step per GPU, far larger than the 126 MB L2, so every step
streams from HBM (no L2 flush needed).

N > 1 (torchrun, one process per GPU): weak scaling -- every GPU owns its own bank of
65 536 voices (voices are independent units: no data-path collective); the only exchange
is the all-reduce of the [T][1][64] mix bus, issued asynchronously so it overlaps the
next step's kernel.  Time = max over ranks, device-timed with CUDA events.  The strong-scaling
configuration of SURVEY 8(d) (ONE 65 536-voice bank, V/G voices per GPU) is measured in the same
run and reported under `other_scaling` (or as the headline with --scaling strong).

After the timed region the last step's output rows of a deterministic 1 024-voice sample are
bit-compared with the CPU checker (`parity`); a mismatch makes the run exit non-zero.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "voice_samples_per_sec"
UNIT = "voice-samples/s"
N_VOICES = 65536
N_BLOCKS = 64
BLOCK = 64


def dist_env():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML during the timed region."""

    def __init__(self, index: int, period_s: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.stop_flag = threading.Event()
        self.sm, self.reasons, self.sm_max, self.power = [], set(), None, []
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self.stop_flag.is_set():
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        if not self.ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_max": max(self.power) if self.power else None}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own SSE implementation on the host cores


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cgroup_cpu_quota():
    """CPU bandwidth limit of this container as (string, cores or None): sched_getaffinity does not
    see a cgroup quota, so the thread count that is actually fastest is found by a sweep (below)."""
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().strip()
            if path.endswith("cpu.max"):
                q, per = txt.split()
                return txt, (None if q == "max" else float(q) / float(per))
            q = float(txt)
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read().strip())
            return txt, (None if q < 0 else q / per)
        except Exception:
            continue
    return "unknown", None


def thread_candidates():
    n = host_threads()
    return sorted({t for t in (16, 32, 64, 128, n) if 1 <= t <= n} | {n})


def reference_chain_runner(n_voices: int, n_blocks: int, repeats: int = 1):
    """Returns (run_once(nthreads) -> seconds, kind).  One call = `repeats` passes over
    n_voices x n_blocks of config A with the compiled reference's own functors (oracle/_ref,
    struct Voice{SineGen; Lopass}) on `nthreads` host threads; falls back to the plain-C port
    (oracle/_port) only where the reference library was never built."""
    from madronalib_b200 import workloads as wl
    from oracle import bindings

    w = wl.config_a(n_voices)
    inp = w.inputs(n_blocks)  # [T][1][V][64]
    if bindings.ref_available():
        R = bindings.RefOracle()
        coef3 = np.ascontiguousarray(w.coef[0:3])
        gain = np.ascontiguousarray(w.coef[3])
        phase = np.ascontiguousarray(w.state[0]).copy()
        ic = np.ascontiguousarray(w.state[1:3]).view(np.float32).copy()
        x = np.ascontiguousarray(inp[:, 0])

        def run_once(nthreads):
            _, sec = R.chain_sine_lopass_gain(x, coef3, gain, phase, ic, nthreads, repeats)
            return sec
        return run_once, "reference"
    if not os.path.exists(bindings.PORT_LIB):
        bindings.build("port")
    P = bindings.PortOracle()

    def run_once(nthreads):
        t0 = time.perf_counter()
        for _ in range(repeats):
            P.run(w.spec, n_voices, n_blocks, inp, w.state, w.coef, nthreads=nthreads)
        return time.perf_counter() - t0
    return run_once, "port"


def best_thread_count(run_once):
    """Untimed set-up: one warm call, then the best of two calls per candidate thread count."""
    run_once(host_threads())  # page faults, thread start
    sweep = {}
    for nt in thread_candidates():
        sweep[nt] = min(run_once(nt), run_once(nt))
    best = min(sweep, key=sweep.get)
    return best, {str(k): round(v * 1e3, 2) for k, v in sweep.items()}


REF_VOICES = 32768  # bounded sample: half the bank (2 x 0.5 GB host buffers), same per-voice work
REF_REPEATS = 4     # passes per step inside one thread launch (amortises thread start-up)


def cpu_baseline(budget_s: float = 10.0):
    """Time the reference chain on a bounded sample of the same workload (best thread count of a sweep)."""
    V = REF_VOICES
    run_once, kind = reference_chain_runner(V, N_BLOCKS, REF_REPEATS)
    nthreads, sweep = best_thread_count(run_once)
    secs, t_start = [], time.perf_counter()
    while len(secs) < 3 or (time.perf_counter() - t_start < budget_s and len(secs) < 40):
        secs.append(run_once(nthreads))
    vs = V * N_BLOCKS * BLOCK * REF_REPEATS
    med = float(np.median(secs))
    quota, _ = cgroup_cpu_quota()
    return {"value": vs / med, "unit": UNIT, "cores": nthreads, "kind": kind,
            "sample": f"{V} voices x {N_BLOCKS} blocks x {REF_REPEATS} passes per call, {len(secs)} calls "
                      f"of config A (median call {med * 1e3:.1f} ms), std::thread x {nthreads}",
            "thread_sweep_ms_per_call": sweep, "host_threads_visible": host_threads(), "cgroup_cpu_max": quota}


def run_reference_arm(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    V, reps = REF_VOICES, REF_REPEATS
    run_once, kind = reference_chain_runner(V, N_BLOCKS, reps)
    nthreads, sweep = best_thread_count(run_once)
    t = run_once(nthreads)
    # keep the whole run within a few minutes: shrink the per-step sample if needed
    total_steps = args.steps + args.warmup
    while t * total_steps > 150.0 and (reps > 1 or V > 1024):
        if reps > 1:
            reps //= 2
        else:
            V //= 2
        run_once, kind = reference_chain_runner(V, N_BLOCKS, reps)
        t = run_once(nthreads)
    for _ in range(args.warmup):
        run_once(nthreads)
    secs = [run_once(nthreads) for _ in range(args.steps)]
    vs = V * N_BLOCKS * BLOCK * reps
    total = float(np.sum(secs))
    value = vs * args.steps / total
    quota, _ = cgroup_cpu_quota()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config A: SineGen->Lopass(SVF)->gain, contract R, 48 kHz; "
                               f"bounded sample {V} voices x {N_BLOCKS} blocks x {reps} passes per step "
                               "(same per-voice work as the 65536-voice bank; the reference's Bank loop is "
                               "independent per voice)",
                   "voices": V, "blocks_per_step": N_BLOCKS * reps},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": kind,
                         "sample": f"{V} voices x {N_BLOCKS} blocks x {reps} passes per step, "
                                   f"{args.steps} steps",
                         "thread_sweep_ms_per_call": sweep, "host_threads_visible": host_threads(),
                         "cgroup_cpu_max": quota},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------
# this repo's arm


def parity_check(w, sel, n_steps, T, inp_sel, got_rows, got_state):
    """Outside every timed region: replay `n_steps` steps of T blocks for the sampled voices `sel`
    on the CPU checker (the compiled reference where oracle/_ref exists, else the port), starting
    from the bank's initial state, and bit-compare the LAST step's output rows and the final state
    words with what the GPU produced for those voices."""
    from oracle import bindings
    if bindings.ref_available():
        O, kind = bindings.RefOracle(), "reference (oracle/_ref)"
    else:
        if not os.path.exists(bindings.PORT_LIB):
            bindings.build("port")
        O, kind = bindings.PortOracle(), "port (oracle/_port)"
    coef = np.ascontiguousarray(w.coef[:, sel])
    st = np.ascontiguousarray(w.state[:, sel])
    nt = host_threads()
    out = None
    for _ in range(n_steps):
        out, _, st = O.run(w.spec, len(sel), T, inp_sel, st, coef, nthreads=nt)
    a, b = np.ascontiguousarray(got_rows).view(np.uint32), out[:, 0].view(np.uint32)
    bad_rows = int(np.any(a != b, axis=(0, 2)).sum())
    bad_state = int(np.any(np.ascontiguousarray(got_state) != st, axis=0).sum())
    return {"rows": int(len(sel)), "blocks": int(T), "steps_replayed": int(n_steps),
            "mismatches": bad_rows + bad_state, "row_mismatches": bad_rows, "state_mismatches": bad_state,
            "checker": kind}


def contract_e_legs(torch, api, wl, w, V, T, args, n_e2e, h_out, h_mix, vs_per_step):
    """Contract E through mlb_synth_process_host (pinned event records in), with a bit-compare of 64 sampled
    voices against the CPU checker (port bank -> port / reference graph) outside the timed regions."""
    res = {}
    prm = wl.synth_bank_params(V)
    ev_np = wl.synth_events(V, T)
    h_ev = torch.empty(ev_np.nbytes, dtype=torch.uint8).pin_memory()
    h_ev.numpy()[:] = ev_np.view(np.uint8).reshape(-1)
    ev = h_ev.numpy().view(ev_np.dtype).reshape(T, V)
    bank = api.VoiceBank(48000.0, *prm)
    g = api.VoiceGraph(w.spec, V, api.FLAG_FAST if args.fast else api.FLAG_EXACT)
    try:
        g.set_coefs(w.coef)
        g.set_state(w.state)
        calls = 0
        for name, want_out in (("contract_E", True), ("contract_E_mix", False)):
            o = h_out.numpy() if want_out else None
            g.process_events_host(bank, ev, want_out=want_out, want_mix=True, out=o, mix=h_mix)
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                g.process_events_host(bank, ev, want_out=want_out, want_mix=True, out=o, mix=h_mix)
            dt = time.perf_counter() - t0
            calls += 1 + n_e2e
            res[name] = {"value": vs_per_step * n_e2e / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / n_e2e,
                         "h2d_bytes_per_step": int(ev.nbytes),
                         "d2h_bytes_per_step": int((h_out.numel() * 4 if want_out else 0) + h_mix.nbytes),
                         "time_chunks": g.last_host_slices,
                         "kernels": "voice_bank_kernel (kPitch row) -> " + g.kernel_name,
                         "path": "mlb_synth_process_host (pinned event records; rows stay in HBM)"}
            if want_out and not args.no_parity:
                from oracle import bindings
                sel = np.linspace(0, V - 1, 64).astype(np.int64)
                rows, _ = bindings.port_voice_bank().run(48000.0, *(p_[sel] for p_ in prm),
                                                         np.ascontiguousarray(np.tile(ev[:, sel], (calls, 1))))
                O = bindings.RefOracle() if bindings.ref_available() else bindings.PortOracle()
                want, _, _ = O.run(w.spec, len(sel), T * calls, np.ascontiguousarray(rows[:, 0:1]),
                                   np.ascontiguousarray(w.state[:, sel]), np.ascontiguousarray(w.coef[:, sel]))
                a = np.ascontiguousarray(h_out.numpy()[:, 0][:, sel]).view(np.uint32)
                b = want[T * (calls - 1):, 0].view(np.uint32)
                res[name]["parity"] = {"rows": int(len(sel)), "blocks": int(T), "steps_replayed": int(calls),
                                       "mismatches": int(np.any(a != b, axis=(0, 2)).sum())}
    finally:
        g.close()
        bank.close()
    return res


class Leg:
    """One bank on this rank (weak: the whole 65 536-voice bank; strong: this rank's V/G shard)."""

    def __init__(self, torch, api, wl, dist, dev, V_bank, v0, v1, T, fast, use_mix, collective="peer"):
        self.torch, self.api, self.dist = torch, api, dist
        full = wl.config_a(V_bank)
        self.full = full
        self.v0, self.v1, self.V, self.T = v0, v1, v1 - v0, T
        self.w = full if (v0 == 0 and v1 == V_bank) else wl.Workload(
            full.name, full.spec, v1 - v0, np.ascontiguousarray(full.coef[:, v0:v1]),
            np.ascontiguousarray(full.state[:, v0:v1]))
        self.graph = api.VoiceGraph(self.w.spec, self.V, api.FLAG_FAST if fast else api.FLAG_EXACT)
        self.graph.set_coefs(self.w.coef)
        self.graph.set_state(self.w.state)
        self.h_in = torch.empty((T, 1, self.V, BLOCK), dtype=torch.float32).pin_memory()
        full.inputs(T, v0=v0, v1=v1, out=self.h_in.numpy())
        self.d_in = self.h_in.to(dev, non_blocking=True)
        self.d_out = torch.empty((T, 1, self.V, BLOCK), dtype=torch.float32, device=dev)
        self.use_mix = use_mix
        self.d_mix = [torch.zeros((T, 1, BLOCK), dtype=torch.float32, device=dev) for _ in range(2)]
        from madronalib_b200.parallel import MixBusReducer, PeerMixBus
        # the mix-bus all-reduce: "peer" = fused into the kernel that finishes the local sum, over NVLink peer
        # memory (no collective call per step); "nccl" = the checked fallback, issued asynchronously
        self.peer = None
        self.collective = "none"
        if dist is not None and use_mix:
            self.collective = collective
            if collective in ("peer", "peer-sync"):
                # "peer": the exchange (write to peers, wait for their rows, sum) on the bus's own stream so that it
                # overlaps the next step like an async NCCL all-reduce; "peer-sync": all in the step's kernel.
                # Should CUDA IPC be unavailable on a box, every rank falls back to NCCL together and says so.
                err = None
                try:
                    self.peer = PeerMixBus(dist, api, self.graph, T * BLOCK, async_completion=(collective == "peer"))
                except Exception as e:  # noqa: BLE001 -- reported in the JSON line, never silent
                    err = repr(e)
                flag = self.torch.tensor([0 if err is None else 1], dtype=self.torch.int32, device=dev)
                dist.all_reduce(flag)
                if int(flag.item()) != 0:
                    if self.peer is not None:
                        self.peer.close()
                        self.peer = None
                    self.collective = "nccl (peer-memory mix bus unavailable: %s)" % (err or "failed on another rank")
        self.reducer = MixBusReducer(dist if (self.peer is None and self.collective.startswith("nccl")) else None)
        # the reduction of the mix partials (and the multi-GPU exchange behind it) runs on the graph's own stream,
        # beside the next step's kernel; d_mix is double-buffered and the timed region ends with mix_wait (drain).
        # Not with NCCL: its all-reduce has to be ordered after the finished local mix on the caller's stream.
        self.mix_async = bool(use_mix and not self.collective.startswith("nccl") and
                              not os.environ.get("MLB_BENCH_SYNC_MIX"))
        if self.mix_async:
            self.graph.set_mix_async(True)
        self.steps_done = 0
        self.stream = torch.cuda.current_stream()

    def step(self, i):
        m = self.d_mix[i & 1]
        self.reducer.wait(i)  # the all-reduce issued two steps ago on this buffer
        self.graph.process_device(self.d_in, self.d_out, m if self.use_mix else None, self.T,
                                  self.stream.cuda_stream)
        if self.use_mix:
            self.reducer.submit(i, m)  # all-reduce of the [T][1][64] mix bus, overlaps step i+1
        self.steps_done += 1

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def drain(self):
        self.reducer.drain()
        if self.peer is not None or self.mix_async:
            self.graph.mix_wait(self.stream.cuda_stream)

    def timed(self, steps, warmup, sampler=None):
        """W untimed warm-up steps, then exactly `steps` steps bracketed by barrier + synchronize;
        device time (CUDA events on the launching stream), max over ranks."""
        torch = self.torch
        for i in range(warmup):
            self.step(i)
        self.drain()
        self.barrier()
        launches0 = self.api.kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler:
            sampler.start()
        self.barrier()
        e0.record(self.stream)
        for i in range(steps):
            self.step(i)
        self.drain()
        e1.record(self.stream)
        self.barrier()
        if sampler:
            sampler.stop_flag.set()
            sampler.join()
        launches = self.api.kernel_launches() - launches0
        ms = e0.elapsed_time(e1)
        if self.dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device=self.d_out.device)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    def parity(self, n_rows=1024):
        """Bit-compare a deterministic sample of voice rows of the most recent step with the CPU checker."""
        n = min(n_rows, self.V)
        sel = np.unique(np.concatenate([np.linspace(0, self.V - 1, n).astype(np.int64), [0, self.V - 1]]))
        idx = self.torch.from_numpy(sel).to(self.d_out.device)
        rows = self.d_out[:, 0].index_select(1, idx).cpu().numpy()
        st = self.graph.get_state()[:, sel]
        inp_sel = np.ascontiguousarray(self.h_in.numpy()[:, :, sel])
        return parity_check(self.w, sel, self.steps_done, self.T, inp_sel, rows, st)

    def dump_outputs(self, path, steps, n_rows=2048, max_bytes=60 << 20):
        """Write what the last step returned to its caller: the output rows of a fixed, seeded sample of voices
        (out_rows.npy [T][n][64], their indices in out_rows_voices.npy) and the mix bus (mix.npy [T][64]).
        The sample shrinks for long steps so that the rows stay under `max_bytes` (the whole dump under 64 MB).
        Must run before anything else launches the graph again."""
        os.makedirs(path, exist_ok=True)
        n = max(1, min(n_rows, self.V, max_bytes // (self.T * BLOCK * 4)))
        sel = np.sort(np.random.default_rng(0).choice(self.V, n, replace=False))
        idx = self.torch.from_numpy(sel).to(self.d_out.device)
        np.save(os.path.join(path, "out_rows.npy"), self.d_out[:, 0].index_select(1, idx).cpu().numpy())
        np.save(os.path.join(path, "out_rows_voices.npy"), sel.astype(np.float64))
        if self.use_mix:
            np.save(os.path.join(path, "mix.npy"), self.d_mix[(steps - 1) & 1][:, 0].cpu().numpy())  # as step() picks it

    def detach_collective(self):
        """Local mix only from here on (used to measure what the collective costs)."""
        if self.peer is not None:
            self.peer.close()
            self.peer = None
        self.reducer = type(self.reducer)(None)
        self.collective = "none"

    def close(self):
        if self.peer is not None:
            self.peer.close()
            self.peer = None
        self.graph.close()


def run_cuda_arm(args):
    import torch

    from madronalib_b200 import api, workloads as wl

    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible; this repo has no CPU fallback "
                         "(use --impl reference for the CPU reference arm)")
    torch.cuda.set_device(local_rank)
    api.init(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    nccl_warm = 0
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29513")
        dist.init_process_group("nccl", rank=rank, world_size=world,
                                device_id=torch.device("cuda", local_rank))
        # NCCL sets its channels up lazily during the first collectives: warm it up on its own,
        # untimed and outside the W warm-up steps (which stay exactly as given)
        nccl_warm = 20
        dummy = torch.zeros((args.blocks, 1, BLOCK), dtype=torch.float32, device=dev)
        for _ in range(nccl_warm):
            dist.all_reduce(dummy)
        torch.cuda.synchronize()

    V, T = args.voices, args.blocks
    use_mix = bool(args.mix)
    strong = args.scaling == "strong"
    if strong:
        v0, v1 = V * rank // world, V * (rank + 1) // world
    else:
        v0, v1 = 0, V
    leg = Leg(torch, api, wl, dist, dev, V, v0, v1, T, args.fast, use_mix, args.collective)
    graph = leg.graph
    collective = leg.collective
    torch.cuda.synchronize()

    sampler = ClockSampler(physical_gpu_index(local_rank)) if rank == 0 else None
    ms, launches = leg.timed(args.steps, args.warmup, sampler)
    if args.dump_outputs and rank == 0:
        leg.dump_outputs(args.dump_outputs, args.steps)
    vs_per_step = leg.V * T * BLOCK
    vs_job = (V if strong else V * world) * T * BLOCK
    value = vs_job * args.steps / (ms * 1e-3)

    # ---- parity of what was just timed (outside the timed region): the last step's rows ----
    par = leg.parity() if not args.no_parity else None
    if par is not None and dist is not None:
        t = torch.tensor([par["mismatches"]], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        par["mismatches_all_ranks"] = int(t.item())

    # ---- what the collective costs: the same K steps with the bus detached (local mix only) ----
    collective_cost = None
    if world > 1 and use_mix:
        leg.detach_collective()
        ms_local, _ = leg.timed(args.steps, 1)
        collective_cost = {"kind": collective, "ms_per_step_with": ms / args.steps,
                           "ms_per_step_local_mix_only": ms_local / args.steps,
                           "us_per_step": 1e3 * (ms - ms_local) / args.steps}

    # ---- roofline of the dominant kernel: per-launch CUDA-event durations (library events on
    # the launching stream), measured live, outside the timed region above ----
    kms = []
    for i in range(min(args.steps, 20)):
        graph.process_device(leg.d_in, leg.d_out, leg.d_mix[0] if use_mix else None, T, leg.stream.cuda_stream)
        kms.append(graph.last_kernel_ms())
    kernel_ms = float(np.mean(kms))
    n_groups = (leg.V + 31) // 32
    # SURVEY 8(d): freq row in + output row out = 8 B per voice-sample, plus per launch and voice the
    # state read+written (2 x 12 B), 3 coefficients and the gain (16 B).  The kernel's own mix-bus
    # scratch (one 256-B partial per 32-voice group and block, written once) is NOT algorithmic: it is
    # reported on its own line.
    alg_bytes = 2 * leg.V * T * BLOCK * 4 + leg.V * (2 * 3 * 4 + 4 * 4)
    scratch_bytes = T * n_groups * BLOCK * 4 if use_mix else 0
    peak, peak_src = measured_peak_gbs()
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "kernel": graph.kernel_name, "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": alg_bytes,
                "bytes_per_voice_sample": alg_bytes / vs_per_step,
                "mix_scratch_bytes_per_launch": scratch_bytes,
                "whole_step_frac": alg_bytes / (ms / args.steps * 1e-3) / 1e9 / peak}
    traffic_file = os.path.join(ROOT, "profiles", "traffic_latest.json")
    if os.path.exists(traffic_file) and leg.V == N_VOICES and T == N_BLOCKS:
        try:
            with open(traffic_file) as f:
                tj = json.load(f)
            roofline["traffic"] = tj.get("dram_bytes_per_launch")
            roofline["traffic_source"] = tj.get("source")  # an ncu capture of a named build, not of this run
        except Exception:
            pass

    # ---- e2e: the same step through the reference-facing C-ABI call with HOST buffers:
    # pinned host in -> H2D -> kernel -> D2H -> pinned host out, all inside the timed call ----
    h_out = torch.empty((T, 1, leg.V, BLOCK), dtype=torch.float32).pin_memory()
    h_mix = np.empty((T, 1, BLOCK), np.float32)
    n_e2e = max(1, min(args.steps, args.e2e_steps if world == 1 else 2))
    graph.process_host(leg.h_in.numpy(), T, want_out=True, want_mix=use_mix, out=h_out.numpy(), mix=h_mix)
    leg.barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        graph.process_host(leg.h_in.numpy(), T, want_out=True, want_mix=use_mix, out=h_out.numpy(),
                           mix=h_mix)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t_e2e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        e2e_s = float(t_e2e.item())
    e2e = {"value": vs_job * n_e2e / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(leg.h_in.numel() * 4),
           "d2h_bytes_per_step": int(h_out.numel() * 4 + (h_mix.nbytes if use_mix else 0)),
           "steps": n_e2e, "host_slices": graph.last_host_slices,
           "path": "mlb_graph_process_host (pinned host buffers, contract R)"}

    # ---- other I/O contracts of the same chain through the same host entry point (SURVEY 8d):
    # S = per-voice scalar frequency (DSPVector(float) broadcast, examples/audio-and-midi/sine.cpp:33)
    #     in, per-voice rows out;  M = scalar frequency in, mix bus out only (Synth::processVector).
    # Reported beside the graded contract-R e2e, never as a fraction of the HBM roofline.
    variants = {}
    if not args.no_variants and world == 1:
        from madronalib_b200.graph import GraphSpec, SINE_ZERO_PHASE
        w = leg.w
        gs = GraphSpec()
        pf = gs.param()
        ps = gs.node("SINE", pf)
        plp = gs.node("LOPASS", ps)
        pk = gs.param()
        gs.output(gs.node("MULTIPLY", plp, pk))
        coef_s = gs.new_coefs(V)
        coef_s[0] = wl.base_freq(V)
        coef_s[1:4] = w.coef[0:3]
        coef_s[4] = w.coef[3]
        st_s = gs.new_state(V)
        st_s[0] = SINE_ZERO_PHASE
        graph_s = api.VoiceGraph(gs, V, api.FLAG_FAST if args.fast else api.FLAG_EXACT)
        graph_s.set_coefs(coef_s)
        graph_s.set_state(st_s)
        for name, want_out in (("contract_S", True), ("contract_M", False)):
            graph_s.process_host(None, T, want_out=want_out, want_mix=True,
                                 out=h_out.numpy() if want_out else None, mix=h_mix)
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                graph_s.process_host(None, T, want_out=want_out, want_mix=True,
                                     out=h_out.numpy() if want_out else None, mix=h_mix)
            dt = time.perf_counter() - t0
            variants[name] = {"value": vs_per_step * n_e2e / dt, "unit": UNIT,
                              "h2d_bytes_per_step": 0,
                              "d2h_bytes_per_step": int((h_out.numel() * 4 if want_out else 0) + h_mix.nbytes),
                              "kernel": graph_s.kernel_name}
        graph_s.close()
        # E = event records in (72 B per voice and vector; EventsToSignals::processVector on the device,
        #     MLEventsToSignals.cpp:383-470), the kPitch row feeding the SAME fused chain as its frequency row
        #     without leaving HBM, per-voice rows (+ mix bus) out;  E_mix = events in, mix bus out only
        #     (Synth::processVector, MLSynth.h:36-60).  mlb_synth_process_host, time-chunked on three streams.
        try:
            variants.update(contract_e_legs(torch, api, wl, w, V, T, args, n_e2e, h_out, h_mix, vs_per_step))
        except Exception as ex:  # a reported side leg: its failure must not lose the graded line
            variants["contract_E"] = {"error": repr(ex)}
    del h_out

    # ---- the other scaling mode of SURVEY 8(d) beside the headline one (N > 1 only): weak = every GPU
    # its own 65 536-voice bank; strong = ONE 65 536-voice bank, V/G voices per GPU.  Same step
    # protocol (kernel + mix-bus all-reduce), same timing rules, own parity block. ----
    other = None
    if world > 1 and not args.no_other_scaling:
        kernel_name = graph.kernel_name
        leg.close()
        del leg.d_in, leg.d_out, leg.h_in
        if strong:
            leg2 = Leg(torch, api, wl, dist, dev, V, 0, V, T, args.fast, use_mix, args.collective)
        else:
            leg2 = Leg(torch, api, wl, dist, dev, V, V * rank // world, V * (rank + 1) // world, T, args.fast,
                       use_mix, args.collective)
        torch.cuda.synchronize()
        ms2, launches2 = leg2.timed(args.steps, args.warmup)
        vs_job2 = (V * world if strong else V) * T * BLOCK
        par2 = leg2.parity() if not args.no_parity else None
        if par2 is not None:
            t = torch.tensor([par2["mismatches"]], dtype=torch.int64, device=dev)
            dist.all_reduce(t)
            par2["mismatches_all_ranks"] = int(t.item())
        other = {"scaling": "weak" if strong else "strong", "value": vs_job2 * args.steps / (ms2 * 1e-3),
                 "unit": UNIT, "ms_per_step": ms2 / args.steps, "steps": args.steps, "warmup": args.warmup,
                 "voices_per_gpu": leg2.V, "voices_total": V * world if strong else V,
                 "gpu_launches": int(launches2), "kernel": leg2.graph.kernel_name, "parity": par2,
                 "collective": leg2.collective}
        leg2.detach_collective()
        ms2l, _ = leg2.timed(args.steps, 1)
        other["collective_cost"] = {"kind": other["collective"], "ms_per_step_with": ms2 / args.steps,
                                    "ms_per_step_local_mix_only": ms2l / args.steps,
                                    "us_per_step": 1e3 * (ms2 - ms2l) / args.steps}
        leg2.close()
    else:
        kernel_name = graph.kernel_name
        leg.close()

    line = None
    rc = 0
    if rank == 0:
        cpu = cpu_baseline() if (world == 1 and not args.no_cpu_baseline) else None
        mode = "strong" if strong else "weak"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": mode, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": "config A: 65536-voice SineGen->Lopass(SVF)->gain, 48 kHz, contract R "
                            "(per-voice freq rows in, per-voice rows out, [T][V][64] f32), "
                            + ("exact (bit-identical to the reference SSE path)" if not args.fast
                               else "fast (FMA contraction allowed)"),
                "voices_per_gpu": leg.V, "voices_total": V if strong else V * world,
                "blocks_per_step": T, "samples_per_block": BLOCK,
                "mix_bus": use_mix,
                "mix_reduce": "asynchronous (own stream, overlaps the next step; joined before the timed region ends)"
                              if leg.mix_async else "on the step's stream",
                "parallelism": f"voices x{world} ({mode}), mix-bus all-reduce ({collective})"
                               + (f"; NCCL warmed up by {nccl_warm} untimed collectives before the "
                                  f"{args.warmup} warm-up steps" if world > 1 else ""),
                "l2": "inputs+outputs %.2f GB per step and GPU >> 126 MB L2 (no flush needed)"
                      % (2 * leg.V * T * BLOCK * 4 / 1e9),
                "kernel": kernel_name,
            },
            "roofline": roofline, "e2e": e2e, "e2e_other_contracts": variants,
            "gpu_launches": int(launches),
            "clocks": sampler.summary() if sampler else None,
            "realtime_x": value / ((V if strong else V * world) * 48000.0),
            "parity": par,
        }
        if collective_cost is not None:
            line["collective_cost"] = collective_cost
        if other is not None:
            line["other_scaling"] = other
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    bad = 0
    for p_ in (par, other["parity"] if other else None, variants.get("contract_E", {}).get("parity")):
        if p_ is not None:
            bad += p_.get("mismatches_all_ranks", p_["mismatches"])
    if bad:
        sys.stderr.write(f"bench.py: PARITY FAILURE: {bad} sampled voice rows differ from the CPU checker\n")
        rc = 3
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--voices", type=int, default=N_VOICES,
                    help="voices per GPU (weak scaling) or in total (strong scaling)")
    ap.add_argument("--blocks", type=int, default=N_BLOCKS)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = 65536 voices per GPU (default, the line's `value`); strong = 65536 "
                         "voices in total, V/G per GPU (SURVEY 8d).  The other mode is measured in the same run "
                         "and reported under `other_scaling`.")
    ap.add_argument("--collective", default="peer", choices=["peer", "peer-sync", "nccl"],
                    help="N > 1: how the mix bus is all-reduced: peer = inside the kernel over NVLink peer memory "
                         "(default), nccl = torch.distributed all_reduce issued asynchronously")
    ap.add_argument("--mix", type=int, default=1)
    ap.add_argument("--fast", action="store_true", help="allow FMA contraction (not bit-exact)")
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the contract S / M e2e legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the bit-comparison with the CPU checker")
    ap.add_argument("--no-other-scaling", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs (a seeded sample of up to 2048 voice "
                         "rows, at most 64 MB in all, and the mix bus) to DIR as .npy files")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes what the CUDA path computed; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_cuda_arm(args)


if __name__ == "__main__":
    sys.exit(main())
