#!/usr/bin/env python3
"""bench.py -- committed slots/sec of the quorum-vote hot path on B200.

Workload (BASELINE.json configs[1], "cfg2"): MultiPaxos, 5 acceptors (f=2),
thrifty quorum of 3, 2^20 slots in flight per GPU per step.  One STEP is one
pass of the hot path over one window of 2^20 fresh slots:
    3*2^20 Phase2a at the acceptors (ballot CAS + vote cells + Phase2b stream),
    arm 2^20 (slot, round) at the proxy leader  ->  3*2^20 shuffled Phase2b at
    the proxy leader (tally + quorum check + ordered Chosen stream) with the
    co-located replica's log + chosen watermark in the same launch (+ when N > 1
    the new frontier stored into every peer GPU's table over NVLink by that
    kernel: fpx_exchange_*).  One C call per step: fpx_step_dev.
`value` times K steps with every input already resident in HBM (distinct
buffers per step, > L2 in total, fresh state region per step);
`e2e` times steps through the asynchronous host-pointer C ABI (fpx_step_submit /
fpx_step_wait) from pinned host buffers: H2D of the Phase2a and Phase2b batches,
D2H of the Phase2b and Chosen replies, double-buffered.

`--dump-outputs DIR` writes what the last timed step returned to its caller as
DIR/<name>.npy (dump_outputs), so that two builds can be compared output for
output: every input is generated from fixed seeds.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SLOTS_PER_STEP = 1 << 20
CFG = dict(f=2, num_acceptor_groups=1, acceptors_per_group=5, flexible=False, num_leaders=3, num_replicas=3)
Q = CFG["f"] + 1
# Algorithmic bytes per committed slot (SURVEY.md 8(d) / DESIGN.md):
#   acceptor kernel  40*Q  = read 16Q (Phase2a) + write 8Q (vote cell) + write 16Q (Phase2b)
#   tally kernels    16Q+24 = read 16Q (Phase2b) + 8+8 slot state RMW + write 8 (Chosen)
B_ACCEPTOR = 40 * Q
B_TALLY = 16 * Q + 24
B_TALLY_FUSED = B_TALLY + 8 + 8   # + the co-located replica: log put (8) and first-hole scan (8)
B_SLOT = B_ACCEPTOR + B_TALLY
N_BASE = 4  # distinct base traces; step s uses base s % N_BASE re-based onto its own slot window


def config_dict(n_gpus):
    """`config` of the JSON line: identical for the GPU arm and the reference arm."""
    nrec = Q * SLOTS_PER_STEP
    return {"workload": "cfg2: MultiPaxos f=2, 5 acceptors, thrifty quorum 3, 2^20 slots in flight "
                        "per GPU per step, Phase2b globally shuffled",
            "slots_per_step_per_gpu": SLOTS_PER_STEP, "records_per_step_per_gpu": 2 * nrec + SLOTS_PER_STEP,
            "sharding": f"slot % {n_gpus}", "l2": "distinct input buffers and a fresh state window every "
                                                 "step (inputs+state touched per step 196 MB > L2)",
            "bytes_per_slot_algorithmic": B_SLOT}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample-slots", type=int, default=SLOTS_PER_STEP)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra keys (cfg5 on the same GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the reply streams and watermark of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    return args


DUMP_ROWS = 1 << 20   # rows kept per stream over all ranks: float64 Phase2b + Chosen rows come to 48 MB


def dump_outputs(out_dir, rank, n_gpus, r, d_out_p2b, d_out_chosen, d_wm):
    """What the last timed step returned to its caller: the Phase2b and Chosen streams in emission order, the
    watermark and the counts fpx_sync reported.  The workload draws no Nack (main asserts n_nack == 0), so the
    Nack stream is empty and only its count is kept.  float64, because slot numbers outgrow float32's 24-bit
    mantissa.  A stream longer than DUMP_ROWS / n_gpus rows is stored as a fixed seeded sample of its rows, kept
    in stream order.  With N > 1 every rank writes its own files (<name>_rank<r>.npy)."""
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_ROWS // n_gpus

    def rows(t, n):
        a = t[:n].cpu().numpy().astype(np.float64)
        if n > cap:
            a = a[np.sort(np.random.Generator(np.random.PCG64(n)).choice(n, cap, replace=False))]
        return a

    out = {"phase2b": rows(d_out_p2b, r.n_p2b), "chosen": rows(d_out_chosen, r.n_chosen),
           "watermark": d_wm.cpu().numpy().astype(np.float64),
           "sync": np.array([r.status, r.n_p2b, r.n_nack, r.n_chosen, r.watermark], dtype=np.float64)}
    suffix = "" if n_gpus == 1 else f"_rank{rank}"
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the
    committed ncu --set full capture (profiles/r2b_traffic.json); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2b_traffic.json")) as f:
            k = json.load(f)[kernel]
        return int(k["dram_bytes_read"] + k["dram_bytes_write"])
    except Exception:
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------- CPU arms (oracle port)
_CPU_TRACES = {}


def cpu_run(sample_slots, threads):
    """The reference's path restated on the CPU (oracle/fpx_oracle.cc, std::map /
    std::set like the Scala collections), `threads` proxy-leader/acceptor
    partitions by slot % threads (the reference's own scale-out), one pass over a
    bounded sample of the cfg2 workload.  Returns slots/s."""
    from frankenpaxos_b200 import traces as T
    from oracle import fpx_oracle_py as O
    key = (sample_slots, threads)
    if key not in _CPU_TRACES:      # the trace is generated once; only the handlers are timed
        a, p, b = T.workload(12345, CFG, sample_slots)
        _CPU_TRACES[key] = [(a[a["slot"] % threads == t], p[p["slot"] % threads == t], b[b["slot"] % threads == t])
                            for t in range(threads)]
    parts = _CPU_TRACES[key]
    oras = [O.MultiPaxos(CFG["f"], 1, 5, False, 3, 3) for _ in range(threads)]
    done = [0] * threads

    def work(t):
        o, (aa, pp, bb) = oras[t], parts[t]
        o.arm(aa)
        st, _, pb, nk = o.acceptor_phase2a(pp)
        st, _, c = o.proxyleader_phase2b(bb)
        o.replica_chosen(c)
        done[t] = len(c)

    t0 = time.perf_counter()
    if threads == 1:
        work(0)
    else:
        th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        [x.start() for x in th]
        [x.join() for x in th]
    dt = time.perf_counter() - t0
    assert sum(done) == sample_slots
    return sample_slots / dt, dt


def reference_arm(args, rank):
    """--impl reference: the reference's own CPU path.  The Scala/JVM reference
    cannot run (no JVM on the box, no offline build), so this is the C++ oracle
    PORT of the same handlers with the reference's data structures, on all host
    cores via the reference's own partitioning (slot % P)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, 64))
    sample = args.cpu_sample_slots
    vals = []
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_run(min(sample, 1 << 15), threads)
    t_total = 0.0
    for _ in range(args.steps):
        v, dt = cpu_run(sample, threads)
        vals.append(v)
        t_total += dt
        if t_total > 120:
            break
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "committed slots/sec (simulated) at 1M in-flight slots",
        "value": value, "unit": "slots/s", "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup,
        "ms_per_step": 1e3 * sample / value, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": config_dict(args.gpus),
        "cpu_baseline": {"value": value, "unit": "slots/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} slots x {len(vals)} passes, slot % {threads} partitions, "
                                   "C++ oracle port (JVM reference not runnable offline)"},
        "e2e": {"value": value, "unit": "slots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Polls NVML while the timed region runs (it is far shorter than nvidia-smi's
    sampling period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.active = index, [], False, False
        self.max_mhz, self.ok = 0, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample_now(self):
        """One sample.  (Sampling from the launch loop itself was tried: an NVML query costs ~0.1 ms of
        host time and showed up 1:1 in the step time, so the polling thread stays the only sampler; when
        it is starved of the GIL during the short timed region, summary() falls back to a wider window.)"""
        if not self.ok:
            return
        nv = self.nv
        try:
            mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) \
                if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.samples.append((time.perf_counter(), mhz, reasons))
        except Exception:
            pass

    def run(self):
        while self.ok and not self.stop_flag:
            self.sample_now()
            time.sleep(0.0001)

    def summary(self, windows):
        """windows: [(name, t0, t1)] in preference order; the first one holding >= 3 samples is used."""
        chosen, name = [], None
        for nm, t0, t1 in windows:
            chosen = [(m, r) for (t, m, r) in self.samples if t0 <= t <= t1]
            name = nm
            if len(chosen) >= 3:
                break
        if not self.ok or not chosen:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz or None, "reasons": ["unsampled"]}
        self_samples = chosen
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        seen = set()
        for _, r in self_samples:
            for bit, nm in names.items():
                if r & bit:
                    seen.add(nm)
        mhz = sorted(m for m, _ in self_samples)
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(seen),
                "samples": len(mhz), "window": name}


# --------------------------------------------------------------------------- our arm
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from frankenpaxos_b200 import P2A, P2B, CHOSEN, NACK, Engine
    from frankenpaxos_b200 import traces as T

    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device; the product has no CPU path")
    # stdout carries ONE line, the JSON record: whatever native libraries write to fd 1 meanwhile (NCCL prints its
    # version there at any NCCL_DEBUG level >= VERSION) goes to stderr; the record is written to the real stdout
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    N = world
    if args.gpus != N and world == 1 and args.gpus > 1:
        sys.exit("bench.py: launch N>1 with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if N > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"     # stdout carries ONE line: the JSON record
        dist.init_process_group("nccl", device_id=dev)

    K, W = args.steps, max(args.warmup, 3)
    S = K + W
    KI = min(K, 20)          # instrumented steps (CUDA events around every kernel): per-kernel durations
    KE = min(K, 10)          # e2e steps: PCIe-bound and ~12x longer each, a bounded sample keeps the run short
    SE = KE + W
    total_windows = S + KI + (0 if args.no_e2e else SE)
    if total_windows * SLOTS_PER_STEP * N >= (1 << 31):
        sys.exit(f"bench.py: (steps+warmup)*2^20*N must stay below 2^31 slots (int32 slot numbers)")
    n_slots_local = total_windows * SLOTS_PER_STEP
    eng = Engine(slot_capacity=n_slots_local * N, max_batch=Q * SLOTS_PER_STEP, overflow_capacity=1 << 10,
                 device=local_rank, shard_index=rank, shard_count=N, **CFG)
    ext = torch.cuda.ExternalStream(eng.stream, device=dev)
    if N > 1:
        # one global log, slot % N shards: every engine's watermark publication is stored into every peer's
        # frontier table over NVLink by the publishing kernel itself (include/fpx.h, fpx_exchange_*)
        from frankenpaxos_b200 import sharding
        sharding.connect(eng)

    # ---- traces: N_BASE distinct seeded base traces on window 0; step s re-bases onto window s
    base = [T.workload(1000 * rank + b, CFG, SLOTS_PER_STEP) for b in range(N_BASE)]

    def rebase(rec, field, window):
        out = rec.copy()
        local = out[field].astype(np.int64) + window * SLOTS_PER_STEP
        out[field] = (local * N + rank).astype(np.int32)
        return out

    def step_inputs(window):
        a, p, b = base[window % N_BASE]
        return rebase(a, "slot", window), rebase(p, "slot", window), rebase(b, "slot", window)

    def to_dev(rec):
        t = torch.from_numpy(rec.view(np.int32).reshape(len(rec), -1))
        return t.to(dev, non_blocking=False)

    d_arm, d_p2a, d_p2b = [], [], []
    for s in range(S + KI):
        a, p, b = step_inputs(s)
        d_arm.append(to_dev(a)); d_p2a.append(to_dev(p)); d_p2b.append(to_dev(b))
    nrec = Q * SLOTS_PER_STEP
    d_out_p2b = torch.empty((nrec, 4), dtype=torch.int32, device=dev)
    d_out_nack = torch.empty((nrec, 2), dtype=torch.int32, device=dev)
    d_out_chosen = torch.empty((nrec, 2), dtype=torch.int32, device=dev)
    d_wm = torch.zeros(1, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def step(s, ring_slot=-1):
        # one C call = one step of the co-located roles: acceptor batch, arm batch, tally + replica + watermark
        # (+ the exchange: the tally's last CTA stores the new frontier into every peer's table)
        eng.step_dev(d_arm[s].data_ptr(), SLOTS_PER_STEP, d_p2a[s].data_ptr(), nrec, d_out_p2b.data_ptr(),
                     d_out_nack.data_ptr(), d_p2b[s].data_ptr(), nrec, d_out_chosen.data_ptr(), d_wm.data_ptr(), ring_slot)

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for s in range(W):
        step(s)
    r = eng.sync()
    assert r.n_chosen == SLOTS_PER_STEP and r.n_nack == 0, (r.n_chosen, r.n_nack)

    sampler = ClockSampler(local_rank)
    sampler.start()
    e_begin, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = eng.launch_count
    barrier()
    t_timed0 = time.perf_counter()
    e_begin.record(ext)
    for k in range(K):
        step(W + k)
    e_end.record(ext)
    barrier()
    t_timed1 = time.perf_counter()
    launches = eng.launch_count - launches0
    ms = e_begin.elapsed_time(e_end)
    r = eng.sync()
    assert r.status == 0 and r.n_chosen == SLOTS_PER_STEP and r.n_nack == 0
    exp_wm = (S * SLOTS_PER_STEP) * N + rank
    assert r.watermark == exp_wm, (r.watermark, exp_wm)
    if args.dump_outputs:    # before the instrumented pass reuses the output buffers
        dump_outputs(args.dump_outputs, rank, N, r, d_out_p2b, d_out_chosen, d_wm)
    global_prefix = None
    if N > 1:   # every shard's frontier after step S, as the peers stored it into THIS rank's table
        global_prefix, fr = eng.global_watermark(epoch=S)
        assert fr.tolist() == [(S * SLOTS_PER_STEP) * N + g for g in range(N)], fr
        assert global_prefix == (S * SLOTS_PER_STEP) * N

    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if N > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = N * K * SLOTS_PER_STEP / (ms_max * 1e-3)

    # ---- per-kernel durations: a second, instrumented pass (CUDA events between the kernels cost ~5 us
    # each on the stream, so they stay out of the pass that produces `value`)
    e_i0, e_i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_i0.record(ext)
    for k in range(KI):
        step(S + k, ring_slot=k)
    e_i1.record(ext)
    eng.sync()
    kms = np.array([eng.step_kernel_ms(k) for k in range(KI)])
    acc_ms, tally_ms = float(kms[:, 0].mean()), float(kms[:, 1].mean())
    arm_ms = float(np.mean([eng.step_arm_ms(k) for k in range(KI)]))
    peak, peak_src = peaks()
    acc_gbs = B_ACCEPTOR * SLOTS_PER_STEP / (acc_ms * 1e-3) / 1e9
    tally_gbs = B_TALLY_FUSED * SLOTS_PER_STEP / (tally_ms * 1e-3) / 1e9

    # ---- e2e: the asynchronous host-pointer step (fpx_step_submit / fpx_step_wait), pinned host buffers,
    # every input copied H2D and every reply stream copied D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        h_in = []
        for s in range(SE):
            a, p, b = step_inputs(S + KI + s)
            h_in.append(tuple(torch.from_numpy(x.view(np.int32).reshape(len(x), -1)).pin_memory() for x in (p, b)))
        h_out = [(torch.empty((nrec, 4), dtype=torch.int32).pin_memory(), torch.empty((nrec, 2), dtype=torch.int32).pin_memory(),
                  torch.empty((nrec, 2), dtype=torch.int32).pin_memory()) for _ in range(2)]

        def submit(s):
            p, b = h_in[s]
            o1, o2, o3 = h_out[s & 1]
            # arm = NULL: the proxy leader arms from the Phase2a batch it forwards (one upload, not two)
            eng.step_submit(None, 0, p.data_ptr(), nrec, b.data_ptr(), nrec, o1.data_ptr(), o2.data_ptr(), o3.data_ptr())

        def wait(s):
            n1, n2, n3, wm = eng.step_wait()
            assert n1 == nrec and n2 == 0 and n3 == SLOTS_PER_STEP, (n1, n2, n3)
            return wm

        def e2e_run(first, count):
            submit(first)
            for s in range(first + 1, first + count):
                submit(s)          # H2D of step s overlaps the kernels and the D2H of step s-1
                wait(s - 1)
            return wait(first + count - 1)

        e2e_run(0, W)
        barrier()
        t0 = time.perf_counter()
        wm_last = e2e_run(W, KE)
        barrier()
        dt = time.perf_counter() - t0
        assert wm_last == ((S + KI + SE) * SLOTS_PER_STEP) * N + rank, wm_last
        assert h_out[(SE - 1) & 1][2][:SLOTS_PER_STEP, 0].min().item() >= ((S + KI + SE - 1) * SLOTS_PER_STEP) * N
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if N > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": N * KE * SLOTS_PER_STEP / float(t.item()), "unit": "slots/s", "steps": KE,
               "h2d_bytes_per_step": 2 * 16 * nrec, "d2h_bytes_per_step": 16 * nrec + 8 * SLOTS_PER_STEP + 160,
               "ms_per_step": 1e3 * float(t.item()) / KE,
               "api": "fpx_step_submit + fpx_step_wait (host pointers, pinned; double-buffered: H2D of step k+1 "
                      "overlaps kernels and D2H of step k; the arm batch is the Phase2a batch)"}
    sampler.stop_flag = True
    t_all1 = time.perf_counter()
    clocks = sampler.summary([("timed region", t_timed0, t_timed1),
                              ("timed region + instrumented + e2e regions (timed region too short to sample 3 times)",
                               t_timed0, t_all1)])
    eng.close()
    del d_arm, d_p2a, d_p2b
    torch.cuda.empty_cache()

    extra = {}
    if not args.no_extra:
        # the extra keys never cost the headline line: a failure is reported in place (every rank runs the same
        # deterministic code, so they fail or pass together)
        try:
            extra["cfg5"] = cfg5_extra(torch, dist, dev, rank, N, local_rank)
        except Exception as e:   # noqa: BLE001
            extra["cfg5"] = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0:
            try:
                extra["cfg4"] = cfg4_extra(torch, dev, local_rank)
            except Exception as e:   # noqa: BLE001
                extra["cfg4"] = {"error": f"{type(e).__name__}: {e}"}

    cpu = None
    if rank == 0 and N == 1:
        v, dt = cpu_run(args.cpu_sample_slots, 1)
        cpu = {"value": v, "unit": "slots/s", "cores": 1, "kind": "port",
               "sample": f"{args.cpu_sample_slots} slots of the cfg2 workload, one pass ({dt:.1f} s), "
                         "single-threaded C++ oracle port of the Scala handlers (JVM reference not runnable offline)"}

    if rank == 0:
        step_ms = ms_max / K
        dominant = "tally_kernel" if tally_ms >= acc_ms else "acceptor_phase2a_kernel"
        kern = {"acceptor_phase2a_kernel": {"ms": acc_ms, "GB/s": acc_gbs, "frac": acc_gbs / peak,
                                            "algorithmic_bytes_per_launch": B_ACCEPTOR * SLOTS_PER_STEP,
                                            "traffic": ncu_traffic("acceptor_phase2a_kernel")},
                "tally_kernel": {"ms": tally_ms, "GB/s": tally_gbs, "frac": tally_gbs / peak,
                                 "algorithmic_bytes_per_launch": B_TALLY_FUSED * SLOTS_PER_STEP,
                                 "traffic": ncu_traffic("tally_kernel"),
                                 "note": "ProxyLeader.handlePhase2b + the co-located replica's handleChosen and the "
                                         "first-hole scan in one launch: 16Q+24 (tally) + 8 (log put) + 8 (scan) B/slot"},
                "arm_kernel": {"ms": arm_ms}}
        line = {
            "metric": "committed slots/sec (simulated) at 1M in-flight slots",
            "value": value, "unit": "slots/s", "n_gpus": N, "steps": K, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": config_dict(N),
            # the dominant kernel by time of the step (CUDA events of the instrumented pass)
            "roofline": {"bound": "hbm", "kernel": dominant, "achieved": kern[dominant]["GB/s"], "peak": peak,
                         "unit": "GB/s", "frac": kern[dominant]["frac"], "traffic": kern[dominant]["traffic"],
                         "algorithmic_bytes_per_launch": kern[dominant]["algorithmic_bytes_per_launch"],
                         "ms_per_launch": kern[dominant]["ms"], "peak_source": peak_src,
                         "timing": f"CUDA events on the engine's stream around every kernel of {KI} instrumented steps "
                                   "run right after the timed region (events between kernels cost ~5 us each, so the "
                                   "pass that produces `value` carries none)"},
            "kernels": dict(kern, **{"whole_step_GB/s": B_SLOT * SLOTS_PER_STEP / (step_ms * 1e-3) / 1e9,
                                     "whole_step_frac": B_SLOT * SLOTS_PER_STEP / (step_ms * 1e-3) / 1e9 / peak}),
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "exchange": None if N == 1 else {"kind": "peer-mapped NVLink stores from the tally kernel's last CTA into "
                                                    "every shard's frontier table (fpx_exchange_*), no collective launch",
                                             "global_prefix_after_timed_region": global_prefix},
            "extra": extra,
        }
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if N > 1:
        dist.destroy_process_group()


def cfg4_extra(torch, dev, local_rank, n_instances=1 << 20, f=2, reps=3):
    """BASELINE configs[3]: EPaxos, 5 replicas, 20 % key-conflict rate, 2^20 instances, as replica 0 sees them:
    device time of each handler batch on device-resident rows (fpx_epaxos_*_dev, CUDA events on the handle's
    stream, best of `reps` fresh replicas) with its algorithmic bytes per message."""
    from frankenpaxos_b200 import traces as T
    from frankenpaxos_b200.epaxos import EpaxosReplica
    n = 2 * f + 1
    lead, pa, ok = T.epaxos_cfg4(0, f=f, n_instances=n_instances, me=0)
    td = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32)).to(dev)
    d_lead, d_pa, d_ok = td(lead), td(pa), td(ok)
    d_rep = torch.zeros((len(pa), 4 + n), dtype=torch.int32, device=dev)
    d_ev = torch.zeros((len(ok), 2 + n), dtype=torch.int32, device=dev)
    best, counts = {}, None
    for _ in range(reps):
        eng = EpaxosReplica(f, 0, n_instances // n + 2, max_batch=1 << 20, device=local_rank)
        ext = torch.cuda.ExternalStream(eng.stream, device=dev)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(ext); eng.lead_dev(d_lead.data_ptr(), len(lead))
        e[1].record(ext); eng.preaccept_dev(d_pa.data_ptr(), len(pa), d_rep.data_ptr())
        e[2].record(ext); eng.preacceptok_dev(d_ok.data_ptr(), len(ok), d_ev.data_ptr())
        e[3].record(ext)
        eng.sync()
        for name, j in (("lead", 0), ("preaccept", 1), ("preacceptok", 2)):
            best[name] = min(best.get(name, 1e9), e[j].elapsed_time(e[j + 1]))
        ev = d_ev.cpu().numpy()
        counts = (int((ev[:, 0] == 1).sum()), int((ev[:, 0] == 2).sum()))
        eng.close()
    msgs = {"lead": len(lead), "preaccept": len(pa), "preacceptok": len(ok)}
    # input row + reply row + cmdLog row read+write (+ the 384-byte leader row for lead; for an Ok the leader
    # row's header, stamp and answer sectors, 32 bytes each)
    alg = {"lead": 4 * (8 + n) + 64 + 384, "preaccept": 4 * (6 + 2 * n) + 4 * (4 + n) + 2 * 64,
           "preacceptok": 4 * (6 + n) + 4 * (2 + n) + 3 * 32}
    peak, _ = peaks()
    return {"config": "cfg4: EPaxos n=5 f=2, 2^20 instances, BernoulliSingleKeyWorkload(0.2), replica 0's view, "
                      "device-resident rows", "fast_commits": counts[0], "slow_paths": counts[1],
            "calls": {k: {"messages": msgs[k], "kernel_ms": best[k], "messages_per_s": msgs[k] / (best[k] * 1e-3),
                          "algorithmic_bytes_per_message": alg[k], "GB/s": alg[k] * msgs[k] / (best[k] * 1e-3) / 1e9,
                          "frac": alg[k] * msgs[k] / (best[k] * 1e-3) / 1e9 / peak} for k in best}}


def cfg5_extra(torch, dist, dev, rank, N, local_rank, K5=4, W5=2):
    """BASELINE configs[4]: vanilla Mencius, 7 servers (f=3), owner = slot % 7, the log sharded slot % N over
    the N GPUs of the box, the chosen prefix exchanged through the engines' frontier tables.  Device-resident
    steps of 2^20 slots per GPU: client requests at the owners (arm + own vote), 6 Phase2a per slot at the
    other servers, 6 shuffled Phase2b per slot tallied, replica log + watermark (+ exchange)."""
    from frankenpaxos_b200 import VANILLA_MENCIUS, Engine
    from frankenpaxos_b200 import traces as T
    cfg, n = T.config_by_name("cfg5")
    f, srv = cfg["f"], cfg["acceptors_per_group"]
    S5 = K5 + W5
    eng = Engine(slot_capacity=S5 * n * N, max_batch=(srv - 1) * n, protocol=VANILLA_MENCIUS, device=local_rank,
                 shard_index=rank, shard_count=N, **cfg)
    if N > 1:
        from frankenpaxos_b200 import sharding
        sharding.connect(eng)
    ext = torch.cuda.ExternalStream(eng.stream, device=dev)
    ins = []
    for s in range(S5):
        req, p, b = T.vanilla_cfg5(500 + 10 * rank + s % 2, f, n, slot_stride=N, slot_offset=rank + s * n * N)
        ins.append(tuple(torch.from_numpy(x.view(np.int32).reshape(len(x), -1)).to(dev) for x in (req, p, b)))
    nrec = (srv - 1) * n
    o_rep = torch.empty((nrec, 4), dtype=torch.int32, device=dev)
    o_ch = torch.empty((nrec, 2), dtype=torch.int32, device=dev)
    wm = torch.zeros(1, dtype=torch.int32, device=dev)

    def step(s):
        dr, dp, db = ins[s]
        # one C call per step: client requests, Phase2a batch, tally + log put + watermark (+ exchange) in one kernel
        eng.vm_step_dev(dr.data_ptr(), n, dp.data_ptr(), nrec, o_rep.data_ptr(), db.data_ptr(), nrec, o_ch.data_ptr(), wm.data_ptr())
    for s in range(W5):
        step(s)
    eng.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if N > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record(ext)
    for k in range(K5):
        step(W5 + k)
    e1.record(ext)
    if N > 1:
        dist.barrier()
    torch.cuda.synchronize()
    r = eng.sync()
    assert r.status == 0 and r.n_chosen == n and r.watermark == S5 * n * N + rank, (r.status, r.n_chosen, r.watermark)
    gp = None
    if N > 1:
        gp, fr = eng.global_watermark(epoch=S5)
        assert gp == S5 * n * N, (gp, fr)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if N > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / K5
    eng.close()
    return {"config": f"cfg5: vanilla Mencius n=7 f=3, owner = slot % 7, log sharded slot % {N}, 2^20 slots per GPU per "
                      "step, 6 Phase2a + 6 Phase2b per slot, both shuffled", "n_gpus": N, "steps": K5, "warmup": W5,
            "ms_per_step": ms, "value": N * n / (ms * 1e-3), "unit": "slots/s",
            "messages_per_s": N * (1 + 2 * (srv - 1)) * n / (ms * 1e-3), "global_prefix": gp,
            "calls": "fpx_vm_step_dev: vm_client_request + vm_phase2a + tally with the log put and the watermark fused (3 launches, device pointers)"}


if __name__ == "__main__":
    main()
