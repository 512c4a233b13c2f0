#!/usr/bin/env python
"""bench.py — consensus reads/sec of the UMI-consensus hot path (BASELINE.json metric).

N=1 workload = BASELINE.json configs[1]: simplex consensus, 10 M families, depth 8, 150 bp,
substitution error rate 1e-3, synthetic (generator: fgumi_b200/synth.py), one B200.
A "step" = one pass of the hot path (ONE kernel launch through fgb_vote_device) over the whole
batch, inputs resident in HBM.  N>1: every rank owns its own 10 M-family shard (families shard
trivially; weak scaling), no data-path collective; the end-of-run device counters are summed with
one NCCL all-reduce.

Keys beyond the base contract:
  roofline      dominant kernel (vote_kernel): algorithmic bytes per launch / CUDA-event time
  cpu_baseline  the CPU oracle (a C++ restatement of fgumi 0.2.0; the Rust reference cannot be
                built here) on a bounded sample, all host threads, rank 0, N=1 only
  e2e           same metric through the host-buffer C-ABI call (fgb_submit/fgb_wait) from pinned
                host memory, H2D + vote + D2H inside the timed region

  e2e_records   the record-level boundary (the reference's `ConsensusCaller`): raw BAM records in pinned
                host memory -> fgb_caller_add_groups + fgb_caller_flush -> ConsensusOutput bytes, beside
                the same host code over the CPU oracle's vote (oracle/libfgb_cpu_caller.so)
  duplex / codec / zipf   device-resident kernel legs for BASELINE configs 3, 4 and 5 (per-kernel ms and
                fraction of the HBM roofline)

`--impl reference` times the reference's CPU algorithm (the oracle built for speed,
oracle/liboracle_native.so, best thread count) on a bounded sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, the consensus columns of the last step for a fixed, seeded
sample of families (rank 0's shard), so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # runs from the tree as build() left it, which may be read-only

METRIC = "consensus reads/sec (simplex 150bp, depth-8 families)"
UNIT = "consensus_reads/s"
DEPTH, READ_LEN, ERR = 8, 150, 1e-3
PARAMS = dict(error_rate_pre_umi=45, error_rate_post_umi=40, min_reads=1,
              min_consensus_base_quality=2)
# --dump-outputs: 16384 families x 150 positions x 4 float32 columns = 39 MB
DUMP_FAMILIES, DUMP_SEED = 16384, 20251017


def algorithmic_bytes(n_units: int, n_reads: int, sum_len: int, sum_cons: int) -> int:
    """SURVEY §8(d): per unit 2*sum(len) in + 6*cons_len out + 8*(n_reads+1) + 8 index bytes."""
    return 2 * sum_len + 6 * sum_cons + 8 * (n_reads + n_units) + 8 * n_units


def dump_outputs(torch, out_dir: str, host_batch, out, dev) -> None:
    """Writes what fgb_vote_device left in `out` for a fixed, seeded sample of families: `base` (ASCII code),
    `qual`, `depth` and `errors` as float32 [families, READ_LEN] arrays, and `family` (float64) the sampled
    families' indices in the batch."""
    n = host_batch.n_units
    fams = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(DUMP_FAMILIES, n), replace=False))
    units = host_batch.units
    assert (units["cons_len"][fams] == READ_LEN).all()
    pos = units["out_off"][fams].astype(np.int64)[:, None] + np.arange(READ_LEN, dtype=np.int64)[None, :]
    idx = torch.from_numpy(pos).to(dev)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "family.npy"), fams.astype(np.float64))
    for name, col in (("base", out.base), ("qual", out.qual), ("depth", out.depth), ("errors", out.errors)):
        a = col[idx].cpu().numpy()
        if a.dtype == np.int16:          # the device holds u16 counts in int16 tensors
            a = a.view(np.uint16)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per launch of vote_kernel from the committed ncu --set full capture, if any."""
    p = os.path.join(ROOT, "profiles", "vote_kernel_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


def cpu_quota() -> int:
    """CPUs this process may actually use: the cgroup CPU quota (cpu.max) capped by the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def bind_to_gpu_numa(torch, local: int):
    """Run this rank (and therefore first-touch its page-locked buffers) on the NUMA node its GPU hangs off.
    Never raises; returns a short description for the bench line."""
    try:
        pr = torch.cuda.get_device_properties(local)
        dev = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read())
        if node < 0:
            return {"node": None, "note": "device reports no NUMA node"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception as e:      # pragma: no cover
        return {"node": None, "note": repr(e)[:80]}


def link_peak(torch, dev, nbytes: int = 1 << 30):
    """Measured host<->device copy bandwidth of this box from page-locked memory (GB/s): the roofline of `e2e`."""
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = {}
    for name, fn in (("h2d_gbs", lambda: d.copy_(h, non_blocking=True)), ("d2h_gbs", lambda: h.copy_(d, non_blocking=True))):
        fn(); torch.cuda.synchronize()
        best = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        out[name] = best
    # both directions at once (the e2e pipeline overlaps the copy back of one chunk with the upload of the next)
    h2 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    s2 = torch.cuda.Stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    d.copy_(h, non_blocking=True)
    with torch.cuda.stream(s2):
        h2.copy_(d, non_blocking=True)
    torch.cuda.current_stream().wait_stream(s2)
    e1.record(); torch.cuda.synchronize()
    out["duplex_gbs_each"] = nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del h, h2, d
    return out


class ClockSampler:
    """`nvidia-smi -lms 20` in the background.  It is started before the warm-up (the tool needs a few
    hundred ms to come up -- longer than a short timed region) and every sample is stamped on arrival;
    begin() / end() bracket the timed region and the summary uses the samples that fall inside it
    (all samples under load -- warm-up included -- if none does).  Never raises."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, cmd=None):
        self.samples = []          # (arrival time, line)
        self.proc = None
        self.index = index
        self.t0 = self.t1 = None
        self.cmd = cmd or ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                           "--format=csv,noheader,nounits", "-lms", "20"]

    def start(self):
        try:
            self.proc = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        try:
            for line in self.proc.stdout:
                self.samples.append((time.perf_counter(), line.strip()))
        except Exception:
            pass

    def wait_ready(self, timeout: float = 2.0):
        """Block (bounded) until the tool has delivered its first sample."""
        try:
            t_end = time.perf_counter() + timeout
            while self.proc and not self.samples and time.perf_counter() < t_end and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            pass

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        try:
            if self.t1 is None:
                self.t1 = time.perf_counter()
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

            def parse(rows):
                mhz, mx, reasons = [], None, set()
                for _, s in rows:
                    f = [x.strip() for x in s.split(",")]
                    if len(f) < 6:
                        continue
                    try:
                        mhz.append(float(f[0])); mx = float(f[1])
                    except ValueError:
                        continue
                    for nm, v in zip(names, f[2:6]):
                        if v.lower().startswith("active"):
                            reasons.add(nm)
                return mhz, mx, reasons
            rows = list(self.samples)
            inside = [r for r in rows if self.t0 is not None and self.t0 - 0.02 <= r[0] <= self.t1 + 0.02]
            mhz, mx, reasons = parse(inside)
            window = "timed region"
            if not mhz:
                mhz, mx, reasons = parse(rows)
                window = "warm-up + timed region"
            return {"sm_mhz": float(np.median(mhz)) if mhz else None, "sm_max_mhz": mx,
                    "reasons": sorted(reasons), "samples": len(mhz), "window": window}
        except Exception as e:      # the clocks line must never cost the bench line
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling failed: %r" % (e,)]}


def _pileup(n_units, depth, L, error_rate, seed, min_input_q=10):
    """fgumi_b200/synth.py host_pileup, restated here so that the CPU arm imports no product code."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    tmpl = acgt[rng.integers(0, 4, size=(n_units, 1, L))]
    bases = np.broadcast_to(tmpl, (n_units, depth, L)).copy()
    if error_rate > 0:
        err = rng.random((n_units, depth, L)) < error_rate
        shift = rng.integers(1, 4, size=(n_units, depth, L))
        code = np.searchsorted(acgt, bases)
        bases = np.where(err, acgt[(code + shift) % 4], bases)
    pos = np.arange(L, dtype=np.float64)
    curve = np.where(pos < 10, 25.0 + (pos / 10.0) * 12.0, 37.0)
    curve = np.where(pos >= 100, np.maximum(37.0 - (pos - 100.0) * 0.08, 2.0), curve)
    q = np.clip(np.rint(curve[None, None, :] + rng.normal(0.0, 2.0, size=(n_units, depth, L))), 2, 41)
    quals = q.astype(np.uint8)
    low = quals < min_input_q
    return np.where(low, np.uint8(ord("N")), bases).astype(np.uint8), np.where(low, np.uint8(2), quals).astype(np.uint8)


def oracle_batch(n_units: int, seed: int = 1234):
    """The CPU arm's input: the SoA batch of include/fgumi_b200.h built with numpy only (no product code is
    imported or loaded by the CPU legs), same generator as the GPU arm."""
    from types import SimpleNamespace
    b, q = _pileup(n_units, DEPTH, READ_LEN, ERR, seed)
    Lp = (READ_LEN + 7) // 8 * 8
    R = n_units * DEPTH
    bases = np.zeros((R, Lp), np.uint8); quals = np.zeros((R, Lp), np.uint8)
    bases[:, :READ_LEN] = b.reshape(R, READ_LEN); quals[:, :READ_LEN] = q.reshape(R, READ_LEN)
    reads = ((np.arange(R, dtype=np.uint64) * np.uint64(Lp)) << np.uint64(16)) | np.uint64(READ_LEN)
    units = np.zeros(n_units + 1, dtype=np.dtype([("out_off", "<u8"), ("read_begin", "<u4"), ("cons_len", "<u4")]))
    units["out_off"] = np.arange(n_units + 1, dtype=np.uint64) * np.uint64(Lp)
    units["read_begin"] = np.arange(n_units + 1, dtype=np.uint32) * np.uint32(DEPTH)
    units["cons_len"][:n_units] = READ_LEN
    return SimpleNamespace(n_units=n_units, n_reads=R, n_out=n_units * Lp, bases=np.pad(bases.reshape(-1), (0, 16)),
                           quals=np.pad(quals.reshape(-1), (0, 16)), reads=np.pad(reads, (0, 2)), units=units)


def best_thread_count(batch, outs, max_threads: int, native: bool = True):
    """The host may expose more logical CPUs than it schedules well (SMT, cgroup quotas): probe a few
    thread counts with one pass each and keep the fastest, so the baseline is the CPU at its best."""
    from tests import oracle_lib as O
    quota = cpu_quota()
    cands = sorted({max(1, max_threads >> k) for k in range(0, 4)} | {1, quota, min(max_threads, 2 * quota)})
    O.simplex_batch(batch, 45, 40, 1, 2, max_threads, outs, native=native)      # first-touch
    rates = {}
    for th in cands:
        t = time.perf_counter()
        O.simplex_batch(batch, 45, 40, 1, 2, th, outs, native=native)
        rates[th] = batch.n_units / (time.perf_counter() - t)
    best = max(rates, key=rates.get)
    return best, {str(k): round(v) for k, v in rates.items()}


def cpu_oracle_rate(n_units: int, threads: int, seed: int = 1234, min_seconds: float = 8.0):
    """Times the CPU oracle (TEST INFRASTRUCTURE used only as the measured baseline) on a sample: the build for
    speed (-O3 -march=x86-64-v3, oracle/Makefile) and, for reference, the plain -O2 build the tests use."""
    from tests import oracle_lib as O
    batch = oracle_batch(n_units, seed)
    outs = O.alloc_outputs(batch)
    threads, probe = best_thread_count(batch, outs, threads)

    def rate(native, secs):
        O.simplex_batch(batch, 45, 40, 1, 2, threads, outs, native=native)    # warm (page faults, thread start)
        reps, t = 0, time.perf_counter()
        while True:
            O.simplex_batch(batch, 45, 40, 1, 2, threads, outs, native=native)
            reps += 1
            dt = time.perf_counter() - t
            if dt >= secs or reps >= 2000:
                return n_units * reps / dt, dt, reps
    v, dt, reps = rate(True, min_seconds)
    v_scalar, _, _ = rate(False, 3.0)
    return v, dt, reps, threads, probe, v_scalar


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = int(os.environ.get("FGB_REF_SAMPLE_UNITS", "400000"))
    from tests import oracle_lib as O
    O.build()
    batch = oracle_batch(n, 1234)
    outs = O.alloc_outputs(batch)
    threads, probe = best_thread_count(batch, outs, threads)
    for _ in range(args.warmup):
        O.simplex_batch(batch, 45, 40, 1, 2, threads, outs, native=True)
    t = time.perf_counter()
    for _ in range(args.steps):
        O.simplex_batch(batch, 45, 40, 1, 2, threads, outs, native=True)
    dt = time.perf_counter() - t
    v = n * args.steps / dt
    sample = (f"{n} families depth {DEPTH} x {READ_LEN} bp per step (same generator as the GPU arm); "
              f"threads probed (families/s): {probe}; cgroup CPU quota {cpu_quota()}")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "simplex consensus, depth 8, 150bp, error-rate 1e-3 "
                               "(BASELINE.json configs[1]), bounded sample", "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": sample + "; oracle = C++ restatement of fgumi 0.2.0 "
                                            "(Rust toolchain absent), -O3 -march=x86-64-v3, std::thread over families"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def bench_records(torch, dist, fg, lib, dev, local, world, rank, args, barrier):
    """Record-level leg (every rank runs it on its own GPU with its share of the host threads; rank 0 reports
    the sum), plus -- on rank 0 at N=1 -- the record-level CPU baseline."""
    from fgumi_b200 import benchlegs
    threads = max(1, cpu_quota() // world)
    barrier()
    r = benchlegs.records_leg(torch, fg, lib, local, args.record_families, threads, steps=max(3, min(args.steps, 6)))
    if world > 1:
        t = torch.tensor([r["value"], r.get("one_caller", {}).get("value", 0.0)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        r["value"] = float(t[0].item())
        r["note"] = f"sum over {world} ranks, {threads} host threads each (cgroup CPU quota {cpu_quota()})"
        # ConsensusCallingStats::merge (caller.rs:278-285): all 24 host counters of the ranks' callers, one all-reduce
        cs = torch.tensor(r.get("caller_stats") or [0] * 24, dtype=torch.int64, device=dev)
        dist.all_reduce(cs, op=dist.ReduceOp.SUM)
        r["caller_stats"] = [int(x) for x in cs.tolist()]
    if rank == 0 and world == 1 and args.cpu_units > 0:
        try:
            r["cpu_baseline"] = benchlegs.records_cpu_baseline(min(args.record_families, 50000), cpu_quota())
        except Exception as ex:       # pragma: no cover
            r["cpu_baseline"] = {"error": repr(ex)[:200]}
    return r


def bench_duplex(torch, dist, fg, dev, local, world, rank, args):
    from fgumi_b200 import benchlegs
    r = benchlegs.duplex_leg(torch, fg, dev, local, int(os.environ.get("FGB_DUPLEX_MOLECULES", "5000000")))
    return _sum_ranks(torch, dist, dev, world, r)


def bench_codec(torch, dist, fg, dev, local, world, rank, args):
    from fgumi_b200 import benchlegs
    r = benchlegs.codec_leg(torch, fg, dev, local, int(os.environ.get("FGB_CODEC_MOLECULES", "2000000")))
    return _sum_ranks(torch, dist, dev, world, r)


def bench_zipf(torch, dist, fg, dev, local, world, rank, args):
    from fgumi_b200 import benchlegs
    r = benchlegs.zipf_leg(torch, fg, dev, local, int(os.environ.get("FGB_ZIPF_FAMILIES", "100000000")), world, rank)
    if world > 1:      # whole job: all families over the slowest rank's time
        t = torch.tensor([r["k1_ms"]], dtype=torch.float64, device=dev)
        n = torch.tensor([float(r["families_this_rank"])], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
        r["value"] = float(n.item()) / (float(t.item()) * 1e-3)
        r["k1_ms_max_over_ranks"] = float(t.item())
    return r


def _sum_ranks(torch, dist, dev, world, r):
    if world > 1:      # weak scaling: every rank runs the same size; the job's rate is the sum
        t = torch.tensor([r["value"]], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        r["value"] = float(t.item())
        r["note"] = f"sum over {world} ranks (per-kernel ms and fractions are rank 0's)"
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fgumi_b200", choices=["fgumi_b200", "reference"])
    ap.add_argument("--units", type=int, default=int(os.environ.get("FGB_BENCH_UNITS", "10000000")),
                    help="families per GPU per step (BASELINE config: 10 M)")
    ap.add_argument("--e2e-units", type=int, default=int(os.environ.get("FGB_E2E_UNITS", "1000000")))
    ap.add_argument("--cpu-units", type=int, default=int(os.environ.get("FGB_CPU_UNITS", "400000")))
    ap.add_argument("--record-families", type=int, default=int(os.environ.get("FGB_RECORD_FAMILIES", "200000")),
                    help="families per batch of the record-level leg")
    ap.add_argument("--no-modes", action="store_true", help="skip the duplex / CODEC / Zipf kernel legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's consensus columns for a seeded sample of "
                         "families (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.dump_outputs and args.impl != "fgumi_b200":
        ap.error("--dump-outputs applies to --impl fgumi_b200")

    if args.impl == "reference":
        run_reference(args)                  # builds and loads oracle/ only: no product code on this arm
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    g.build()
    import fgumi_b200 as fg
    from fgumi_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: fgumi_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    numa = bind_to_gpu_numa(torch, local)        # before any page-locked allocation (first touch = local node)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))

    eng = fg.Engine(device=local, **PARAMS)
    U = args.units
    depths = np.full(U, DEPTH, dtype=np.int64)
    tb = synth.device_batch(torch, dev, depths, READ_LEN, ERR, seed=42 + rank, min_reads=1)
    out = fg.DeviceColumns(tb.host.n_out, dev)
    bstruct, cstruct = tb.struct(), out.struct()
    stream = torch.cuda.current_stream().cuda_stream
    import ctypes as C
    lib = fg.lib.load()

    def step():
        st = lib.fgb_vote_device(eng._h, C.byref(bstruct), C.byref(cstruct), C.c_void_p(stream))
        if st != 0:
            raise fg.lib.FgbError(st, "fgb_vote_device")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clk = ClockSampler(local)
    clk.start()
    clk.wait_ready()
    for _ in range(args.warmup):
        step()
    barrier()
    eng.stats_reset()
    launches0 = eng.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    clk.begin()
    torch.cuda.nvtx.range_push("fgb_timed")
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    # K4: the only collective on the path — sum the device counters across ranks (in place)
    ctr = None
    if world > 1:
        class _DevPtr:   # zero-copy view of the engine's u64[FGB_NCOUNTERS] counter block
            __cuda_array_interface__ = {"shape": (fg.lib.FGB_NCOUNTERS,), "typestr": "<i8",
                                        "data": (eng.stats_device_ptr(), False), "version": 2}
        ctr = torch.as_tensor(_DevPtr(), device=dev)
        dist.all_reduce(ctr, op=dist.ReduceOp.SUM)
    barrier()
    torch.cuda.nvtx.range_pop()
    clk.end()
    clocks = clk.stop()
    total_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    launches = eng.launch_count() - launches0
    stats_all = eng.stats()   # after the all-reduce every rank's block holds the global sums
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, tb.host, out, dev)

    value = U * world * args.steps / (total_ms * 1e-3)
    # ---- roofline of the dominant kernel (one launch per step) ----
    h = tb.host
    abytes = algorithmic_bytes(h.n_units, h.n_reads, h.n_reads * READ_LEN, h.n_units * READ_LEN)
    k_ms = float(np.mean(per_launch_ms))
    achieved = abytes / (k_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak_gbs()
    tr = recorded_traffic()
    traffic = None
    if tr and tr.get("units") and tr.get("dram_bytes_per_launch"):
        traffic = tr["dram_bytes_per_launch"] * (h.n_units / tr["units"])
    roofline = {"bound": "hbm", "kernel": "vote_kernel", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes_per_launch": abytes, "bytes_per_unit": abytes / h.n_units,
                "kernel_ms": k_ms, "peak_source": peak_src}

    # ---- e2e: host-buffer call, pinned host memory, H2D + vote + D2H inside the timed region ----
    e2e = None
    cpu = None
    if True:
        EU = min(args.e2e_units, U)
        hb = synth.make_descriptors(np.full(EU, DEPTH, dtype=np.int64), READ_LEN, 1)
        nb = hb.n_bytes
        pin = lambda n, dt: torch.empty(n, dtype=dt).pin_memory()
        pb, pq = pin(nb + 16, torch.uint8), pin(nb + 16, torch.uint8)
        pb[:nb].copy_(tb.bases[:nb]); pq[:nb].copy_(tb.quals[:nb])
        torch.cuda.synchronize()
        hb.bases = pb.numpy(); hb.quals = pq.numpy()
        ho = fg.HostColumns(pin(hb.n_out, torch.uint8).numpy(), pin(hb.n_out, torch.uint8).numpy(),
                            pin(hb.n_out, torch.int16).numpy().view(np.uint16),
                            pin(hb.n_out, torch.int16).numpy().view(np.uint16))
        preads = pin(len(hb.reads), torch.int64); preads.numpy()[:] = hb.reads.view(np.int64)
        hb.reads = preads.numpy().view(np.uint64)
        esteps = max(3, min(args.steps, 10))

        def timed_e2e(call, tag):
            for _ in range(args.warmup):
                call(); eng.wait()
            barrier()
            t0 = time.perf_counter()
            torch.cuda.nvtx.range_push(tag)
            for _ in range(esteps):
                call(); eng.wait()
            torch.cuda.synchronize()
            torch.cuda.nvtx.range_pop()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return EU * world * esteps / float(tt.item())

        desc_bytes = hb.n_reads * 8 + (hb.n_units + 1) * 16 + len(hb.tiles) * 32
        d2h = hb.n_out * 6
        # (1) the two-column layout (a base byte and a quality byte per observation)
        v_bytes = timed_e2e(lambda: eng.submit(hb, ho), "fgb_e2e_bytes")
        # (2) PACK8: one byte per observation, expanded on the device in front of the vote.  The
        #     host-side encode is part of source-read preparation, like building the rows themselves.
        packed = fg.pack8_encode(hb.bases[:nb], hb.quals[:nb])
        if packed is not None:
            pp = pin(nb + 16, torch.uint8)
            pp.numpy()[:nb] = packed
            ppn = pp.numpy()
            v_pack = timed_e2e(lambda: eng.submit_pack8(hb, ppn, ho), "fgb_e2e_pack8")
            # (2b) PACK8 in, narrow (u8 depth / errors) out: 4 instead of 6 bytes per position back
            ho8 = fg.HostColumns(ho.base, ho.qual, pin(hb.n_out, torch.uint8).numpy(),
                                 pin(hb.n_out, torch.uint8).numpy())
            v_pack8n = timed_e2e(lambda: eng.submit_ex(hb, ho8, packed=ppn, narrow=True), "fgb_e2e_pack8_u8")
            # (2c) the same with the host-side PACK8 encode (fgb_pack8_encode, one host thread) INSIDE the timed region
            def encode_and_submit():
                st = lib.fgb_pack8_encode(hb.bases.ctypes.data, hb.quals.ctypes.data, nb, ppn.ctypes.data)
                if st != 0:
                    raise fg.lib.FgbError(st, "fgb_pack8_encode")
                eng.submit_ex(hb, ho8, packed=ppn, narrow=True)
            v_pack8enc = timed_e2e(encode_and_submit, "fgb_e2e_pack8_encode")
            e2e = {"value": v_pack8n, "unit": UNIT, "h2d_bytes_per_step": int(nb + desc_bytes),
                   "d2h_bytes_per_step": int(hb.n_out * 4), "units_per_step": EU, "steps": esteps,
                   "api": "fgb_submit_ex(FGB_IN_PACK8, FGB_OUT_U8) + fgb_wait (pinned host buffers: "
                          "1 byte per observation in, 4 bytes per consensus position out); rows arrive PACK8-encoded "
                          "(the encode is part of source-read preparation; `pack8_encode_timed` has it inside)",
                   "pack8_encode_timed": {"value": v_pack8enc, "note": "fgb_pack8_encode on ONE host thread per step + the call above"},
                   "pack8_u16": {"value": v_pack, "h2d_bytes_per_step": int(nb + desc_bytes),
                                 "d2h_bytes_per_step": int(d2h), "api": "fgb_submit_pack8 + fgb_wait"},
                   "two_column": {"value": v_bytes, "h2d_bytes_per_step": int(2 * nb + desc_bytes),
                                  "d2h_bytes_per_step": int(d2h), "api": "fgb_submit + fgb_wait"}}
            # (3) BAM4: 4-bit sequence + raw qualities, rows built on the device (forward-strand reads;
            #     the generator's masked bases are (N, Q2), so the min-quality mask leaves them as is).
            #     Informative extra leg: a failure here must not cost the line.
            try:
                from fgumi_b200.engine import RawColumns, RAW_READ_DTYPE, _NIBBLE
                Lp = (READ_LEN + 7) // 8 * 8
                nib = _NIBBLE[hb.bases[:nb]]
                seq4 = pin(nb // 2 + 32, torch.uint8)
                seq4.numpy()[:nb // 2] = (nib[0::2] << 4) | nib[1::2]
                rr = pin((hb.n_reads + 1) * 16, torch.uint8)
                rrv = rr.numpy().view(RAW_READ_DTYPE)
                rrv["src_off"][:hb.n_reads] = np.arange(hb.n_reads, dtype=np.uint64) * np.uint64(Lp)
                rrv["raw_len"][:hb.n_reads] = READ_LEN
                rrv["flags"][:] = 0
                rawc = RawColumns(seq4.numpy(), hb.quals, rrv, int(nb), 10)
                v_bam4 = timed_e2e(lambda: eng.submit_bam4(hb, rawc, ho), "fgb_e2e_bam4")
                e2e["bam4"] = {"value": v_bam4,
                               "h2d_bytes_per_step": int(nb + nb // 2 + hb.n_reads * 16 + desc_bytes),
                               "d2h_bytes_per_step": int(d2h),
                               "api": "fgb_submit_bam4 + fgb_wait (4-bit sequence + raw qualities)"}
            except Exception as ex:   # pragma: no cover
                e2e["bam4"] = {"error": repr(ex)[:200]}
        else:
            e2e = {"value": v_bytes, "unit": UNIT, "h2d_bytes_per_step": int(2 * nb + desc_bytes),
                   "d2h_bytes_per_step": int(d2h), "units_per_step": EU, "steps": esteps,
                   "api": "fgb_submit + fgb_wait (pinned host buffers)"}
        # the link is the roofline of every e2e leg: measured page-locked copy bandwidth of THIS box
        try:
            link = link_peak(torch, dev)
            h2d_rate = e2e["h2d_bytes_per_step"] * e2e["value"] / EU / world / 1e9      # GB/s per GPU
            e2e["link"] = dict(link, numa=numa)
            e2e["roofline"] = {"bound": "pcie h2d", "achieved": h2d_rate, "peak": link["h2d_gbs"], "unit": "GB/s",
                               "frac": h2d_rate / link["h2d_gbs"]}
        except Exception as ex:       # pragma: no cover
            e2e["link"] = {"error": repr(ex)[:200]}
        del pb, pq, ho, preads
    del tb, out, bstruct, cstruct
    torch.cuda.empty_cache()

    # ---- record-level boundary: raw BAM records -> ConsensusOutput bytes ----
    records_leg = None
    try:
        records_leg = bench_records(torch, dist, fg, lib, dev, local, world, rank, args, barrier)
    except Exception as ex:           # pragma: no cover  (an extra leg never costs the line)
        records_leg = {"error": repr(ex)[:300]}
    # ---- BASELINE configs 3, 4, 5: device-resident kernel legs ----
    modes = {}
    if not args.no_modes:
        for name, fn in (("duplex", bench_duplex), ("codec", bench_codec), ("zipf", bench_zipf)):
            try:
                modes[name] = fn(torch, dist, fg, dev, local, world, rank, args)
            except Exception as ex:   # pragma: no cover
                modes[name] = {"error": repr(ex)[:300]}
            torch.cuda.empty_cache()

    if rank == 0 and world == 1 and args.cpu_units > 0:
        os.sched_setaffinity(0, range(os.cpu_count() or 1)) if hasattr(os, "sched_setaffinity") else None   # the CPU arm may use every core
        threads = os.cpu_count() or 1
        v, dtc, reps, threads, probe, v_scalar = cpu_oracle_rate(args.cpu_units, threads)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "logical_cpus": os.cpu_count(), "cpu_quota": cpu_quota(),
               "thread_probe": probe, "kind": "port", "value_O2_generic": v_scalar,
               "sample": f"{reps} passes over {args.cpu_units} families depth {DEPTH} x {READ_LEN} bp, {dtc:.1f} s; "
                         "oracle = C++ restatement of fgumi 0.2.0 (no Rust toolchain) built -O3 -march=x86-64-v3 "
                         "(value_O2_generic: the -O2 build the tests use), std::thread over families"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 in / u8+u16 out, f64 log-likelihood on the exact path",
            "data": "synthetic",
            "config": {"workload": "simplex consensus, 10M families depth=8, 150bp, error-rate 1e-3 "
                                   "(BASELINE.json configs[1])",
                       "families_per_gpu": U, "depth": DEPTH, "read_len": READ_LEN,
                       "error_rate": ERR, "params": "-1 45 -2 40 -m 10 --min-consensus-base-quality 2 "
                                                    "--min-reads 1, overlapping pre-pass off",
                       "parallelism": f"range-shard x{world}",
                       "l2": "inputs (24 GB/GPU) larger than L2; no flush needed"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_records": records_leg,
            "duplex": modes.get("duplex"), "codec": modes.get("codec"), "zipf": modes.get("zipf"),
            "gpu_launches": int(launches), "clocks": clocks,
            "counters": stats_all,
        }
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def _one_line_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version from C on the first
    collective), so file descriptor 1 is pointed at stderr for the whole run and Python's sys.stdout keeps the real
    one: only print() calls of this script reach it."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


if __name__ == "__main__":
    _one_line_stdout()
    main()
