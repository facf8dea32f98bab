#!/usr/bin/env python
"""bench.py — joined rows/sec of the GPU hash join on BASELINE.json config 2 (and its N-GPU shuffled form).

Workload (N = 1): "C2" = 2-table INNER hash join, 100 M build x 1 B probe rows, BIGINT key + 2 INT payloads per
side, every probe row matches exactly once (SURVEY.md §8d).  One step = build (consume + finish) + probe of the
whole probe table.  value = probe rows / step time with inputs resident in HBM; e2e = the same join driven through
the C-ABI with HOST (pinned) buffers, host<->device copies inside the timed region.

N > 1 (weak scaling): every rank holds a 100 M x 1 B shard of an N-times larger join; both sides are hash-
partitioned on the join key (ExecUtils.partition) and exchanged with one NCCL AllToAllv per column over NVLink,
then joined locally — the plan shape of a hash/hash-distributed MPP join.  value = N x 1 B probe rows / max-over-
ranks step time.

`--impl reference` times the reference-shaped CPU path (oracle/, P = min(cores,16) driver threads, 1000-row chunks,
shared CAS chained table) on a bounded sample of the same workload; rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2_BUILD, C2_PROBE = 100_000_000, 1_000_000_000
PROBE_ALG_BYTES = 68  # SURVEY.md §8d: 16 probe row + 4 bucket head + 8 build key + 8 build payload + 32 output row
BUILD_ALG_BYTES = 24  # 16 row read + 8 table write
METRIC = "joined+aggregated rows/sec; achieved HBM GB/s vs peak, at 1/2/4/8 B200"


def c2_workload_name(world: int) -> str:
    base = "C2: inner hash join 100M build x 1B probe, BIGINT key + 2 INT payloads"
    return base + (", 1 GPU" if world == 1 else f" per GPU, both sides hash-shuffled across {world} GPUs (partition-and-push over NVLink)")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=float(os.environ.get("GSQL_BENCH_SCALE", "1.0")),
                    help="fraction of config 2 (testing only; the contract value is 1.0)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the group-by rooflines (C1 / C3 / C5 share) and the Q3 / C5 pipeline entries")
    ap.add_argument("--e2e-batch", type=int, default=125_000_000, help="probe rows per host batch in the e2e leg")
    ap.add_argument("--workload", default="c2", choices=["c2", "q3", "c5"],
                    help="c2 (default, the contract line): BASELINE config 2 join; q3 / c5: BASELINE configs 4 / 5 pipelines")
    ap.add_argument("--slabs", type=int, default=int(os.environ.get("GSQL_BENCH_SLABS", "1")),
                    help="slabs of the pushed side (N > 1): slab k is consumed while slab k+1 crosses NVLink; 1 measured best at N = 2..8 (r02)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's output columns to DIR/<workload>_<name>.npy (float64, a seeded sample "
                         "of at most 2^20 rows per table) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm returns row counts only)")
    return args


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  In-process NVML polling (cheap driver calls) is
    preferred: a `nvidia-smi -lms` loop stalls the GPU for milliseconds per query, which at ~30 ms per step showed up
    as ~4 ms of idle time per step.  GSQL_BENCH_CLOCKS=smi|nvml|off overrides."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index = index
        self.lines = []
        self.proc = None
        self.nvml = None
        self.mode = os.environ.get("GSQL_BENCH_CLOCKS", "nvml")
        self.period = float(os.environ.get("GSQL_BENCH_CLOCKS_PERIOD_MS", "20")) / 1000.0
        self._stop = threading.Event()

    def start(self):
        if self.mode == "off":
            return
        if self.mode == "nvml" and self._start_nvml():
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _start_nvml(self) -> bool:
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            smax = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            reasons_fn(h)
        except Exception:
            return False
        self.nvml = (pynvml, h, smax, reasons_fn)

        def poll():
            while not self._stop.is_set():
                try:
                    sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                    rs = int(reasons_fn(h))
                    self.lines.append((time.time(), sm, rs))
                except Exception:
                    pass
                self._stop.wait(self.period)
        self.t = threading.Thread(target=poll, daemon=True)
        self.t.start()
        return True

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def _stop_nvml(self, t0: float, t1: float):
        self._stop.set()
        self.t.join(timeout=1.0)
        _, _, smax, _ = self.nvml
        sm, reasons = [], set()
        for ts, mhz, rs in self.lines:
            if ts < t0 or ts > t1:
                continue
            sm.append(float(mhz))
            for bit, nm in self.NVML_REASONS.items():
                if rs & bit:
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(smax), "reasons": sorted(reasons), "samples": len(sm),
                "source": f"nvml, {self.period * 1000:.0f} ms period"}

    def stop(self, t0: float, t1: float):
        if self.nvml:
            return self._stop_nvml(t0, t1)
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(index: int):
    """Pin this process (and the pinned buffers it allocates from now on: first touch) to the NUMA node of GPU `index`:
    at N = 8 the r01 end-to-end leg delivered 2.3x one rank's host throughput because ranks copied across sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        import torch
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        if not uuid.startswith("GPU-"):
            uuid = "GPU-" + uuid
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:   # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:120]}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------ reference arm
def host_threads() -> int:
    return max(1, min(os.cpu_count() or 1, 16))  # ExecUtils.getParallelismForLocal: min(cores, 16)


CPU_SAMPLE = (100_000_000, 100_000_000)  # the FULL 100 M-row build side (table size is what the probe's cache misses depend on), 1/10 of the probe rows
_cpu_tables = {}


def cpu_sample(build_rows: int, probe_rows: int, repeats: int = 1):
    """Reference-shaped CPU join (oracle) on a bounded sample; returns (rows/s incl. build, detail dict)."""
    from galaxysql_b200 import synth
    from oracle import oracle as orc
    P = host_threads()
    if (build_rows, probe_rows) not in _cpu_tables:
        _cpu_tables[(build_rows, probe_rows)] = synth.c2_tables_np(build_rows, probe_rows)
    build, probe = _cpu_tables[(build_rows, probe_rows)]
    spec = orc.JoinSpec(orc.JOIN_INNER, [0], [0], [orc.T_INT64])
    best = None
    for _ in range(repeats):
        r = orc.mt_join(spec, [(c, None) for c in probe], [(c, None) for c in build], nthreads=P, chunk_rows=1000)
        assert r["out_rows"] == probe_rows
        t = r["build_s"] + r["probe_s"]
        if best is None or t < best[0]:
            best = (t, r)
    t, r = best
    return probe_rows / t, {"build_s": r["build_s"], "probe_s": r["probe_s"], "threads": P}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sb, sp = CPU_SAMPLE
    times = []
    for i in range(args.warmup + args.steps):
        v, d = cpu_sample(sb, sp)
        if i >= args.warmup:
            times.append(sp / v)
    ms = 1000.0 * sum(times) / len(times)
    value = sp / (ms / 1000.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": c2_workload_name(args.gpus), "build_rows_per_gpu": C2_BUILD, "probe_rows_per_gpu": C2_PROBE, "scale": 1.0},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": host_threads(), "kind": "port",
                         "sample": f"{sb} build x {sp} probe rows per step (the full build side; 1/10 of the probe rows), {host_threads()} threads, "
                                   "1000-row chunks; the reference Java cannot run (no JDK in the image): this is the oracle port in the reference's "
                                   "parallel shape (P = min(cores, 16) drivers, shared CAS chained table)"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from galaxysql_b200 import api, native as N, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        # the AllToAllv is a grouped ncclSend/ncclRecv per peer: give the p2p path all the channels NVLink can use
        os.environ.setdefault("NCCL_MIN_P2P_NCHANNELS", "32")
        os.environ.setdefault("NCCL_MAX_P2P_NCHANNELS", "32")
        os.environ.setdefault("NCCL_P2P_NET_CHUNKSIZE", "4194304")
        dist.init_process_group("nccl", device_id=dev)
    ctx = api.Context(local_rank)
    stream = ctx.torch_stream()
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.tensor(list(api.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        api.comm_init(ctx, world, rank, bytes(uid.cpu().tolist()))
    if args.workload != "c2":
        run_pipeline_workload(args, ctx, stream, world, rank, local_rank, dev)
        if world > 1:
            ctx.lib.gsql_comm_destroy(ctx.ptr)
            dist.destroy_process_group()
        return

    nb = int(C2_BUILD * args.scale)
    npr = int(C2_PROBE * args.scale)
    key_space = nb * world
    # ---- synthetic shard on the device
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    if world == 1:
        perm = torch.randperm(nb, generator=g, device=dev, dtype=torch.int64)
    else:  # rank r holds keys {r, r+W, r+2W, ...} of the global permutation space, shuffled
        g.manual_seed(42 + rank)
        perm = torch.randperm(nb, generator=g, device=dev, dtype=torch.int64) * world + rank
    build, probe = synth.c2_tables_t(nb, npr, dev, key_space=key_space, probe_start=rank * npr, build_perm=perm)
    torch.cuda.synchronize()

    types = [N.T_INT64, N.T_INT32, N.T_INT32]
    out_types = types + types
    tt = {N.T_INT64: torch.int64, N.T_INT32: torch.int32}
    cap = npr if world == 1 else int(npr * 1.02) + 1_000_000
    out_cols = [(torch.empty(cap, dtype=tt[t], device=dev), None) for t in out_types]
    if world > 1:
        from galaxysql_b200 import pipelines
        bcap = int(nb * 1.05) + 1_000_000
        sj = pipelines.ShuffledJoin(ctx, N.JOIN_INNER, types, types, [0], [0], build_capacity=bcap, probe_capacity=cap, nslabs=args.slabs)

    def b(cols):
        return [(c, None) for c in cols]

    state = {"out_rows": 0, "info": None}

    def step_single():
        j = api.HashJoin(ctx, N.JOIN_INNER, types, types, [0], [0], expected_build_rows=nb)
        j.build_consume_ref(b(build))   # device-resident build side: referenced, not copied (gsql_join_build_consume_ref)
        j.build_finish()
        state["out_rows"] = j.probe_into(b(probe), out_cols, cap)
        state["info"] = j.info()
        j.close()

    def step_multi():
        # both sides are split by ExecUtils.partition(key) and written straight into the owning GPU's receive buffer over
        # NVLink (gsql_xchg_push: no staging copy, no NCCL kernel); the build side's table is built from the receive
        # buffer in place, and probe slab k is joined while slab k+1 is still on the wire (pipelines.ShuffledJoin).
        sj.run(b(probe), b(build), out_cols=out_cols, out_capacity=cap)
        state["out_rows"] = sj.last_rows
        state["info"] = sj.last_info

    step = step_multi if world > 1 else step_single

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the sampler is started BEFORE the warm-up so that the timed region follows the warm-up back to back: an idle gap
    # here (there used to be a 0.3 s sleep) lets the GPU drop out of its boost state and the first timed steps pay the ramp
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    ctx.profile(True)
    ctx.profile_reset()
    launches0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.time()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    t1 = time.time()
    ms_total = ev0.elapsed_time(ev1)
    prof = ctx.profile_dump()
    ctx.profile(False)
    launches = ctx.launch_count - launches0

    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        rows_t = torch.tensor([state["out_rows"]], dtype=torch.int64, device=dev)
        dist.all_reduce(rows_t)
        total_out = int(rows_t.item())
    else:
        total_out = state["out_rows"]
    assert total_out == npr * world, (total_out, npr * world)  # every probe row matches exactly once
    ms_step = ms_total / args.steps
    value = npr * world / (ms_step / 1000.0)

    # ---- parity of the last step's output, outside the timed region: an order-independent 64-bit checksum over EVERY
    # output row (probe.key, p1, p2, build.key, b1, b2), all-reduced over the ranks, against the same checksum computed
    # from the inputs (each probe row joined with its build row through the inverse of the build-key permutation).
    # Equal sums <=> the distributed output is the global join's row multiset (up to a 2^-64 collision).
    n_out = state["out_rows"]
    parity = verify_join_checksum(torch, dist, synth, dev, world, rank, nb, npr, probe, out_cols, n_out)
    assert parity["match"], f"join output checksum mismatch: {parity}"
    if args.dump_outputs:
        names = ["probe_key", "probe_p1", "probe_p2", "build_key", "build_b1", "build_b2"]
        dump_outputs(args.dump_outputs, "c2", [(nm, d[:n_out], None) for nm, (d, _) in zip(names, out_cols)], 3, rank, world)

    # ---- roofline of the dominant kernel(s): the probe phase
    probe_kernels = [k for k in prof if "probe" in k or k == "join_scan"]
    probe_ms = sum(prof[k][1] for k in probe_kernels) / args.steps
    probe_rows_rank = n_out
    peak, peak_src = measured_peak_gbs()
    achieved = PROBE_ALG_BYTES * probe_rows_rank / (probe_ms / 1000.0) / 1e9 if probe_ms > 0 else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum per 1 B probe rows of the probe-phase kernels, from this round's committed
    # `ncu --set full` capture (profiles/r02_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep); null when the
    # capture is absent or was taken for another table mode — never a number typed into this file
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        ent = tj.get("radix" if state["info"].partitions > 1 else "one_partition")
        if ent:
            traffic = float(ent["dram_bytes_per_probe_row"]) * probe_rows_rank
    except Exception:
        traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": "+".join(sorted(probe_kernels)), "kernel_ms_per_step": probe_ms,
                "algorithmic_bytes_per_probe_row": PROBE_ALG_BYTES, "peak_source": peak_src,
                "per_kernel_ms_per_step": {k: v[1] / args.steps for k, v in sorted(prof.items())}}

    # ---- e2e: host (pinned) buffers through the C-ABI, rank-local, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, ctx, api, N, build, probe, nb, npr, world, rank, dev, numa)
    # free the big device tables before the CPU leg
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sb, sp = CPU_SAMPLE
        v, d = cpu_sample(sb, sp)
        cpu = {"value": v, "unit": "rows/s", "cores": d["threads"], "kind": "port",
               "sample": f"bounded sample of config 2: {sb} build x {sp} probe rows, {d['threads']} threads, 1000-row chunks "
                         f"(build {d['build_s']:.2f}s + probe {d['probe_s']:.2f}s)"}
    # ---- auxiliary (N = 1 only): the group-by half of the metric on its BASELINE shape, device-resident like `value`.
    # Never allowed to take the headline down: any failure is reported inside the key.
    if not args.no_aux:
        # ---- the rest of the metric inside the same line (the driver keeps `roofline`): the group-by rooflines (N = 1) and
        # the two pipelines BASELINE.json names for 8 GPUs — TPC-H Q3 and the high-cardinality GROUP BY — at this N
        if world > 1:
            sj.close()
        del out_cols, probe, build    # ~50 GB back before the other tables are generated
        torch.cuda.empty_cache()
        if rank == 0 and world == 1:
            for key, fn in (("agg_q1", run_aux_agg), ("agg_c5", run_aux_agg_c5), ("agg_c1", run_aux_agg_c1)):
                try:
                    roofline[key] = fn(ctx, api, N, synth, dev, args.scale, peak)
                except Exception as e:  # noqa: BLE001
                    roofline[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.empty_cache()
        for wl in ("q3", "c5"):
            m = measure_pipeline(args, wl, 3, 2, ctx, stream, world, rank, local_rank, dev)   # collective: every rank takes part
            roofline["pipeline_" + wl] = {"workload": m["config"]["workload"], "rows_per_s": m["value"], "ms_per_step": m["ms_per_step"],
                                          "n_gpus": world, "parity": m["parity"], "stats": m["stats"],
                                          "per_kernel_ms_per_step": m["roofline"]["per_kernel_ms_per_step"]}
            torch.cuda.empty_cache()
    if rank == 0:
        info = state["info"]
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic",
            "config": {"workload": c2_workload_name(world),
                       "build_rows_per_gpu": nb, "probe_rows_per_gpu": npr, "scale": args.scale,
                       "l2": "inputs (16 GB probe per step) are far larger than the 126 MB L2; no explicit flush",
                       "step": "build (consume + finish) + probe of the full probe table" + (" after the key shuffle" if world > 1 else ""),
                       "table_slots": int(info.table_slots), "fast_path": int(info.fast_path), "partitions": int(info.partitions)},
            "roofline": roofline,
            "clocks": clocks,
            "gpu_launches": int(launches),
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.lib.gsql_comm_destroy(ctx.ptr)
        dist.destroy_process_group()


def _mix_rows(torch, key, p1, p2, b1, b2):
    """64-bit mix of one joined row (int64 wraparound arithmetic); summed over rows it is order-independent."""
    from galaxysql_b200 import synth
    h = key * (-7046029254386353131) + p1.to(torch.int64) * (-4658895280553007687) + p2.to(torch.int64) * (-7723592293110705685)
    h = synth.splitmix64_t(h) + b1.to(torch.int64) * 0x2545F4914F6CDD1D + b2.to(torch.int64) * 0x27D4EB2F165667C5
    return synth.splitmix64_t(h)


def verify_join_checksum(torch, dist, synth, dev, world, rank, nb, npr, probe, out_cols, n_out, chunk=1 << 26):
    """Expected: every probe row (key, p1, p2) of this rank joined with THE build row of its key.  Build keys of rank r are
    perm_r * world + r (perm_r = randperm(nb) seeded 42 + r, or seed 42 for world == 1), build payloads are counter-based
    functions of the build row index — so any rank can reconstruct any build row from its key alone."""
    inv = torch.empty(world * nb, dtype=torch.int32, device=dev)
    for r in range(world):
        g = torch.Generator(device=dev)
        g.manual_seed(42 + r if world > 1 else 42)
        perm = torch.randperm(nb, generator=g, device=dev, dtype=torch.int64)
        inv[r * nb:(r + 1) * nb][perm] = torch.arange(nb, dtype=torch.int32, device=dev)
        del perm
    exp = torch.zeros((), dtype=torch.int64, device=dev)
    for lo in range(0, npr, chunk):
        hi = min(npr, lo + chunk)
        k = probe[0][lo:hi]
        i = inv[(k % world) * nb + k // world].to(torch.int64)
        b1 = synth._top31(synth.splitmix64_t(i + (synth.SEED + 1 * synth._STREAM)))
        b2 = synth._top31(synth.splitmix64_t(i + (synth.SEED + 2 * synth._STREAM)))
        exp += _mix_rows(torch, k, probe[1][lo:hi], probe[2][lo:hi], b1, b2).sum()
        del k, i, b1, b2
    del inv
    got = torch.zeros((), dtype=torch.int64, device=dev)
    keys_equal = True
    for lo in range(0, n_out, chunk):
        hi = min(n_out, lo + chunk)
        o = [c[0][lo:hi] for c in out_cols]
        keys_equal = keys_equal and bool((o[0] == o[3]).all())
        got += _mix_rows(torch, o[0], o[1], o[2], o[4], o[5]).sum()
    t = torch.stack([exp, got, torch.tensor(n_out, dtype=torch.int64, device=dev)])
    if world > 1:
        dist.all_reduce(t)
    e, g_, n = (int(v) for v in t.tolist())
    return {"match": bool(e == g_ and n == npr * world and keys_equal), "expected": e, "got": g_, "rows": n,
            "what": "sum over all output rows of mix64(probe.key,p1,p2,b1,b2), all ranks, vs the same sum derived from the inputs"}


DUMP_ROWS = 1 << 20   # rows written per output table and run: at most 6 float64 columns -> 48 MB per dump


def dump_outputs(out_dir, workload, cols, nkey, rank, world, chunk=1 << 26):
    """--dump-outputs: write `cols` ([(name, device values, device nulls | None)], one output table of the last step) as
    out_dir/<workload>_<name>.npy, float64 with NaN for NULL, plus <workload>_rows.npy = [total output rows].

    Row order out of a hash join / group-by is unspecified, so the dump must not depend on it: when the table has more
    than DUMP_ROWS rows, a row is kept when a seeded hash of its first `nkey` columns (the columns that identify it: probe
    row, group key) falls under a threshold, and the kept rows are sorted on all columns.  Two builds that produce the
    same rows therefore write the same arrays.  Every integer these workloads produce is below 2^53, so float64 holds it
    exactly.  With N ranks each rank writes its own share (suffix .rank<r>), DUMP_ROWS / N rows each."""
    import numpy as np
    import torch
    from galaxysql_b200 import synth
    cap = DUMP_ROWS // world
    n = int(cols[0][1].numel())
    threshold = None if n <= cap else int(0.9 * cap / n * (1 << 53))   # ~0.9 * cap rows kept; truncation below never bites
    parts = [[] for _ in cols]
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        f64 = []
        for _, d, nl in cols:
            v = d[lo:hi].to(torch.float64)
            f64.append(v if nl is None else torch.where(nl[lo:hi].bool(), float("nan"), v))
        if threshold is not None:
            h = torch.full((hi - lo,), synth.SEED, dtype=torch.int64, device=f64[0].device)
            for v in f64[:nkey]:
                h = synth.splitmix64_t(h ^ v.view(torch.int64))
            keep = synth._lsr(h, 11) < threshold
            f64 = [v[keep] for v in f64]
        for p, v in zip(parts, f64):
            p.append(v.cpu().numpy())
    arrays = [np.concatenate(p) if p else np.zeros(0) for p in parts]
    order = np.lexsort(arrays[::-1])[:cap]
    suffix = "" if world == 1 else f".rank{rank}"
    os.makedirs(out_dir, exist_ok=True)
    for (name, _, _), a in zip(cols, arrays):
        np.save(os.path.join(out_dir, f"{workload}_{name}{suffix}.npy"), a[order])
    np.save(os.path.join(out_dir, f"{workload}_rows{suffix}.npy"), np.array([n], dtype=np.float64))


def _timed_agg(ctx, make, feed, reps=3):
    """Best wall time of consume+finish over `reps` fresh handles (after one warm-up), and the kernel times of that run."""
    import time as _t
    best, groups, prof_best = None, 0, {}
    for i in range(reps + 1):
        a = make()
        ctx.sync()
        ctx.profile(True)
        ctx.profile_reset()
        t0 = _t.perf_counter()
        feed(a)
        groups = a.finish()
        ctx.sync()
        dt = _t.perf_counter() - t0
        prof = ctx.profile_dump()
        ctx.profile(False)
        a.close()
        if i > 0 and (best is None or dt < best):
            best, prof_best = dt, prof
    return best, groups, prof_best


def _agg_entry(rows, groups, alg_bytes, best_s, prof, peak_gbs, what):
    kern_ms = sum(v[1] for k, v in prof.items() if k.startswith("agg_") and k not in ("agg_slots_init", "agg_state_init", "agg_finalize"))
    top = max(((v[1], k) for k, v in prof.items() if k.startswith("agg_")), default=(0.0, ""))[1]
    gbs = rows * alg_bytes / (kern_ms / 1e3) / 1e9 if kern_ms > 0 else 0.0
    return {"workload": what, "rows": rows, "groups": int(groups), "algorithmic_bytes_per_row": alg_bytes, "ms_wall": best_s * 1e3,
            "rows_per_s": rows / best_s, "kernel_ms": kern_ms, "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs,
            "kernel": top, "per_kernel_ms": {k: v[1] for k, v in sorted(prof.items())}}


def run_aux_agg(ctx, api, N, synth, dev, scale, peak_gbs):
    """BASELINE config 3 shape (TPC-H Q1): 600 M rows, 2 INT keys (3 x 2 values), 8 aggregates over DOUBLE columns,
    44 algorithmic bytes per row (SURVEY.md §8d); one gsql_agg_consume + gsql_agg_finish over device-resident columns."""
    import torch
    n3 = int(600_037_902 * scale)
    flag = synth.rand_i64_t(n3, 4, dev, post=lambda b: synth._u64_mod(b, 3).to(torch.int32))
    status = synth.rand_i64_t(n3, 5, dev, post=lambda b: synth._u64_mod(b, 2).to(torch.int32))
    qty = synth.rand_i64_t(n3, 6, dev, post=lambda b: (synth._u64_mod(b, 50) + 1).to(torch.float64))
    price = synth.rand_i64_t(n3, 7, dev, post=lambda b: (synth._u64_mod(b, 10_410_000) + 90_000).to(torch.float64) / 100.0)
    disc = synth.rand_i64_t(n3, 8, dev, post=lambda b: synth._u64_mod(b, 11).to(torch.float64) / 100.0)
    tax = synth.rand_i64_t(n3, 9, dev, post=lambda b: synth._u64_mod(b, 9).to(torch.float64) / 100.0)
    ship = synth.rand_i64_t(n3, 10, dev, post=lambda b: (synth._u64_mod(b, 2526) + 8036).to(torch.int32))
    cols = [flag, status, qty, price, disc, tax, ship]
    types = [0, 0, 2, 2, 2, 2, 0]
    # the Q1 plan: SUM(qty), SUM(price), SUM(price*(1-disc)), SUM(price*(1-disc)*(1+tax)), AVG(qty), AVG(price), AVG(disc), COUNT(*),
    # l_shipdate <= 1998-09-02 — Project and Filter fused into the aggregation (gsql_agg_spec.derived / row_filter_*)
    aggs = [(N.AGG_SUM, [2]), (N.AGG_SUM, [3]), (N.AGG_SUM, [7]), (N.AGG_SUM, [8]), (N.AGG_AVG, [2]), (N.AGG_AVG, [3]),
            (N.AGG_AVG, [4]), (N.AGG_COUNT_STAR, [])]
    derived = [(N.EXPR_MUL_1MINUS, 3, 4, 0), (N.EXPR_MUL_1MINUS_1PLUS, 3, 4, 5)]
    torch.cuda.synchronize()
    best, groups, prof = _timed_agg(ctx, lambda: api.HashAgg(ctx, types, [0, 1], aggs, 8, derived=derived, row_filter=(6, N.CMP_LE, 10471)),
                                    lambda a: a.consume([(c, None) for c in cols]))
    return _agg_entry(n3, groups, 44, best, prof, peak_gbs, "C3: TPC-H Q1 shape, 600M rows, fused project + filter, 8 aggregates")


def run_aux_agg_c5(ctx, api, N, synth, dev, scale, peak_gbs):
    """One GPU's share of BASELINE config 5 after the shuffle: 500 M rows, 6.25 M distinct BIGINT keys, SUM(double);
    16 algorithmic bytes per row."""
    import torch
    n = int(500_000_000 * scale)
    keys = int(6_250_000 * scale) or 1
    k = synth.rand_i64_t(n, 11, dev, post=lambda b: synth._u64_mod(b, keys) * 8 + 3)
    v = synth.rand_i64_t(n, 12, dev, post=lambda b: synth._lsr(b, 11).to(torch.float64) / float(1 << 53))
    torch.cuda.synchronize()
    best, groups, prof = _timed_agg(ctx, lambda: api.HashAgg(ctx, [N.T_INT64, N.T_FP64], [0], [(N.AGG_SUM, [1])], keys),
                                    lambda a: a.consume([(k, None), (v, None)]))
    return _agg_entry(n, groups, 16, best, prof, peak_gbs, "C5 share: 500M rows, 6.25M distinct keys, SUM(double)")


def run_aux_agg_c1(ctx, api, N, synth, dev, scale, peak_gbs):
    """BASELINE config 1: SELECT k, COUNT(*) FROM t GROUP BY k, 1 M-row INT column, k in [0, 65536); 4 bytes per row."""
    import torch
    n = 1_000_000
    k = synth.rand_i64_t(n, 13, dev, post=lambda b: synth._u64_mod(b, 65536).to(torch.int32))
    torch.cuda.synchronize()
    best, groups, prof = _timed_agg(ctx, lambda: api.HashAgg(ctx, [N.T_INT32], [0], [(N.AGG_COUNT_STAR, [])], 65535),
                                    lambda a: a.consume([(k, None)]), reps=5)
    return _agg_entry(n, groups, 4, best, prof, peak_gbs, "C1: 1M-row INT column, COUNT(*) (launch-bound)")


# ------------------------------------------------------------------------------------------------ q3 / c5 pipelines
def run_pipeline_workload(args, ctx, stream, world, rank, local_rank, dev):
    line = measure_pipeline(args, args.workload, args.steps, args.warmup, ctx, stream, world, rank, local_rank, dev, with_clocks=True,
                            dump_dir=args.dump_outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)


def measure_pipeline(args, workload, steps, warmup, ctx, stream, world, rank, local_rank, dev, with_clocks=False, dump_dir=None):
    """workload q3: BASELINE config 4 (TPC-H Q3, SF300 over 8 GPUs = SF37.5 per GPU, weak scaling);
    --workload c5: BASELINE config 5 (GROUP BY k, SUM(double): 500 M rows and 6.25 M keys per GPU).  One step = the whole
    pipeline of galaxysql_b200/pipelines.py over device-resident tables; value = input rows of all ranks / max step time."""
    import torch
    import torch.distributed as dist
    from galaxysql_b200 import api, native as N, pipelines, synth
    sc = args.scale
    peak, peak_src = measured_peak_gbs()
    if workload == "q3":
        ncust, nord, nline = int(5_625_000 * sc), int(56_250_000 * sc), int(225_000_000 * sc)
        g = torch.Generator(device=dev)
        g.manual_seed(1000 + rank)
        c_custkey = torch.arange(ncust, dtype=torch.int64, device=dev) * world + rank
        c_seg = synth.rand_i64_t(ncust, 20, dev, start=rank * ncust, post=lambda b: synth._u64_mod(b, 5).to(torch.int32))
        o_orderkey = torch.randperm(nord, generator=g, device=dev, dtype=torch.int64) * world + rank
        o_custkey = synth.rand_i64_t(nord, 21, dev, start=rank * nord, post=lambda b: synth._u64_mod(b, ncust * world))
        o_date = synth.rand_i64_t(nord, 22, dev, start=rank * nord, post=lambda b: (synth._u64_mod(b, 2557) + 8035).to(torch.int32))
        o_ship = torch.zeros(nord, dtype=torch.int32, device=dev)
        l_orderkey = synth.rand_i64_t(nline, 23, dev, start=rank * nline, post=lambda b: synth._u64_mod(b, nord * world))
        l_price = synth.rand_i64_t(nline, 24, dev, start=rank * nline, post=lambda b: (synth._u64_mod(b, 10_410_000) + 90_000).to(torch.float64) / 100.0)
        l_disc = synth.rand_i64_t(nline, 25, dev, start=rank * nline, post=lambda b: synth._u64_mod(b, 11).to(torch.float64) / 100.0)
        l_shipd = synth.rand_i64_t(nline, 26, dev, start=rank * nline, post=lambda b: (synth._u64_mod(b, 2557) + 8035).to(torch.int32))
        cust = [(c_custkey, None), (c_seg, None)]
        orders = [(o_orderkey, None), (o_custkey, None), (o_date, None), (o_ship, None)]
        line = [(l_orderkey, None), (l_price, None), (l_disc, None), (l_shipd, None)]
        q3 = pipelines.Q3Pipeline(ctx, customer_capacity=int(ncust * world * 0.25) + 100_000, orders_capacity=int(nord * 0.2) + 100_000,
                                  lineitem_capacity=int(nline * 0.75) + 1_000_000, nslabs=args.slabs, expected_groups=int(nord * 0.1) + 1024)
        state = {}

        def step():
            state["out"] = q3.run(cust, orders, line)

        rows_in = ncust + nord + nline
        what = f"C4: TPC-H Q3 (3-way hash join + group-by), SF{300 * sc / 8:.1f} per GPU x {world} GPUs; customer {ncust} / orders {nord} / lineitem {nline} rows per GPU"
    else:
        n = int(500_000_000 * sc)
        keys = max(int(6_250_000 * sc) * world, 1)
        k = synth.rand_i64_t(n, 30, dev, start=rank * n, post=lambda b: synth._u64_mod(b, keys) * 8 + 3)
        v = synth.rand_i64_t(n, 31, dev, start=rank * n, post=lambda b: synth._lsr(b, 11).to(torch.float64) / float(1 << 53))
        agg = pipelines.TwoPhaseAgg(ctx, [N.T_INT64, N.T_FP64], [0], [(N.AGG_SUM, [1]), (N.AGG_COUNT_STAR, [])], expected_groups=keys,
                                    capacity=int(n * 1.03) + 1_000_000, nslabs=args.slabs, expected_rows=n * world)
        state = {}

        def step():
            state["out"] = agg.run([(k, None), (v, None)])

        rows_in = n
        what = f"C5: GROUP BY k, SUM(double): {n} rows per GPU x {world} GPUs, {keys} distinct keys ({agg.mode} plan)"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0 and with_clocks:
        sampler.start()
    for _ in range(warmup):
        step()
    barrier()
    ctx.profile(True)
    ctx.profile_reset()
    launches0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.time()
    ev0.record(stream)
    for _ in range(steps):
        step()
    ev1.record(stream)
    barrier()
    t1 = time.time()
    ms_total = ev0.elapsed_time(ev1)
    prof = ctx.profile_dump()
    ctx.profile(False)
    launches = ctx.launch_count - launches0
    clocks = sampler.stop(t0, t1) if rank == 0 and with_clocks else None
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / steps
    # ---- parity of the last step's result against a torch restatement of the query on the same tables (outside the timed region)
    out = state["out"]
    if workload == "q3":
        def allgather(t):
            if world == 1:
                return t
            n_ = torch.tensor([t.numel()], dtype=torch.int64, device=dev)
            ns = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
            dist.all_gather(ns, n_)
            m = int(max(int(x.item()) for x in ns))
            pad = torch.zeros(m, dtype=t.dtype, device=dev)
            pad[:t.numel()] = t
            outs = [torch.zeros(m, dtype=t.dtype, device=dev) for _ in range(world)]
            dist.all_gather(outs, pad)
            return torch.cat([o[:int(x.item())] for o, x in zip(outs, ns)])
        building = allgather(c_custkey[c_seg == pipelines.Q3_SEGMENT])
        omask = (o_date < pipelines.Q3_DATE) & torch.isin(o_custkey, building)
        qual = allgather(o_orderkey[omask])
        lmask = (l_shipd > pipelines.Q3_DATE)
        lk = l_orderkey[lmask]
        hit = torch.isin(lk, qual)
        exp_rev = (l_price[lmask][hit] * (1.0 - l_disc[lmask][hit])).sum()
        exp_rows = hit.sum()
        got = torch.stack([out[3][0].sum(), torch.tensor(float(out[0][0].numel()), dtype=torch.float64, device=dev)])
        exp = torch.stack([exp_rev, exp_rows.to(torch.float64)])
        joined_keys = allgather(lk[hit])   # collective: every rank takes part, rank 0 counts the distinct order keys
        exp_groups = torch.tensor([torch.unique(joined_keys).numel() if rank == 0 else 0], dtype=torch.float64, device=dev)
        del joined_keys
        if world > 1:
            dist.all_reduce(got)
            dist.all_reduce(exp)
            dist.all_reduce(exp_groups)
        rel = abs(float(got[0]) - float(exp[0])) / max(abs(float(exp[0])), 1e-300)
        parity = {"match": bool(rel < 1e-9 and int(got[1]) == int(exp_groups[0])), "revenue_rel_err": rel, "groups": int(got[1]),
                  "expected_groups": int(exp_groups[0]), "joined_lineitem_rows": int(exp[1]),
                  "what": "sum of revenue over all groups and number of groups vs a torch restatement (isin / unique) of Q3 on the same tables"}
        stats = q3.stats
    else:
        got = torch.stack([out[1][0].sum(), out[2][0].sum().to(torch.float64), torch.tensor(float(out[0][0].numel()), dtype=torch.float64, device=dev)])
        exp = torch.stack([v.sum(), torch.tensor(float(n), dtype=torch.float64, device=dev)])
        if world > 1:
            dist.all_reduce(got)
            dist.all_reduce(exp)
        rel = abs(float(got[0]) - float(exp[0])) / max(abs(float(exp[0])), 1e-300)
        parity = {"match": bool(rel < 1e-9 and int(got[1]) == int(exp[1]) and int(got[2]) <= keys), "sum_rel_err": rel, "count": int(got[1]),
                  "groups": int(got[2]), "what": "sum of SUM(v) and of COUNT(*) over all groups vs the column totals; groups <= distinct keys"}
        stats = {"mode": agg.mode}
    assert parity["match"], parity
    if dump_dir:
        names = ["l_orderkey", "o_orderdate", "o_shippriority", "revenue"] if workload == "q3" else ["k", "sum_v", "count_star"]
        dump_outputs(dump_dir, workload, [(nm, d, nl) for nm, (d, nl) in zip(names, out)], 3 if workload == "q3" else 1, rank, world)
    (q3 if workload == "q3" else agg).close()
    value = rows_in * world / (ms_step / 1e3)
    return {"metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if workload == "c5" else "int64+f64", "data": "synthetic",
            "config": {"workload": what, "slabs": args.slabs, "scale": sc, "l2": "tables are far larger than the 126 MB L2; no explicit flush"},
            "roofline": {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
                         "per_kernel_ms_per_step": {k_: v_[1] / steps for k_, v_ in sorted(prof.items())}, "peak_source": peak_src},
            "parity": parity, "stats": stats, "clocks": clocks, "gpu_launches": int(launches)}


def run_e2e(args, ctx, api, N, build, probe, nb, npr, world, rank, dev, numa=None):
    """The join as a host caller drives it: pinned host Blocks in, pinned host Blocks out, every copy timed."""
    import torch
    import torch.distributed as dist
    batch = min(args.e2e_batch, npr)
    types = [N.T_INT64, N.T_INT32, N.T_INT32]
    tt = {N.T_INT64: torch.int64, N.T_INT32: torch.int32}
    # host copies of the inputs (pinned) — made once, outside the timed region, like a caller that owns them.  ~22 GB of
    # pinned memory per rank: if any rank cannot get it, every rank skips the leg together (no half-entered collectives)
    ok, hbuild, hprobe, hout = 1, None, None, None
    try:
        hbuild = [torch.empty(nb, dtype=c.dtype, pin_memory=True) for c in build]
        hprobe = [torch.empty(npr, dtype=c.dtype, pin_memory=True) for c in probe]
        hout = [torch.empty(batch if world == 1 else 1, dtype=tt[t], pin_memory=True) for t in types + types]
    except RuntimeError:
        ok = 0
    if world > 1:
        okt = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        ok = int(okt.item())
    if not ok:
        del hbuild, hprobe, hout
        return {"value": None, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "error": "pinned host buffers for the end-to-end leg could not be allocated on every rank"}
    for h, c in zip(hbuild, build):
        h.copy_(c)
    for i, (h, c) in enumerate(zip(hprobe, probe)):
        h.copy_(c)
    torch.cuda.synchronize()

    def view(tensors, lo, hi):
        return [(t[lo:hi].numpy(), None) for t in tensors]

    if world > 1:
        # N > 1: the same work as `value` — upload the rank's shards from pinned host memory, shuffle both sides over NVLink,
        # join, download the joined rows into pinned host memory — every copy inside the timed region
        return run_e2e_multi(args, ctx, api, N, hbuild, hprobe, nb, npr, world, rank, dev, numa, build, probe)

    def step():
        j = api.HashJoin(ctx, N.JOIN_INNER, types, types, [0], [0], expected_build_rows=nb)
        j.build_consume(view(hbuild, 0, nb))
        j.build_finish()
        total = 0
        for lo in range(0, npr, batch):
            hi = min(npr, lo + batch)
            total += j.probe_into(view(hprobe, lo, hi), [(t.numpy(), None) for t in hout], batch)
        j.close()
        return total

    steps = max(1, min(args.steps, 3))
    step()  # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        total = step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    assert total == npr
    h2d = nb * 16 + npr * 16
    d2h = npr * 32
    return {"value": npr * world / dt, "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "numa_binding": numa,
            "ms_per_step": dt * 1000.0, "steps": steps, "probe_batch_rows": batch,
            "path": "gsql_join_build_consume/gsql_join_probe with GSQL_MEM_HOST pinned batches" +
                    (" (every rank joins its own 100M x 1B shard from host memory; probe keys remapped to the rank's key share)" if world > 1 else "")}


def run_e2e_multi(args, ctx, api, N, hbuild, hprobe, nb, npr, world, rank, dev, numa, dbuild, dprobe):
    import torch
    import torch.distributed as dist
    from galaxysql_b200 import pipelines
    types = [N.T_INT64, N.T_INT32, N.T_INT32]
    tt = {N.T_INT64: torch.int64, N.T_INT32: torch.int32}
    cap = int(npr * 1.02) + 1_000_000
    ok, hout = 1, None
    try:
        hq = cap // 4 + 1   # the joined rows leave through a quarter-size pinned buffer, four times (bounds pinned host memory per rank)
        hout = [torch.empty(hq, dtype=tt[t], pin_memory=True) for t in types + types]
    except RuntimeError:
        ok = 0
    okt = torch.tensor([ok], dtype=torch.int32, device=dev)
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    if not int(okt.item()):
        return {"value": None, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "error": "pinned host output buffers could not be allocated on every rank"}
    out_cols = [(torch.empty(cap, dtype=tt[t], device=dev), None) for t in types + types]
    sj = pipelines.ShuffledJoin(ctx, N.JOIN_INNER, types, types, [0], [0], build_capacity=int(nb * 1.05) + 1_000_000, probe_capacity=cap, nslabs=args.slabs)
    st = ctx.torch_stream()

    def step():
        with torch.cuda.stream(st):
            for h, d in zip(hbuild, dbuild):
                d.copy_(h, non_blocking=True)
            for h, d in zip(hprobe, dprobe):
                d.copy_(h, non_blocking=True)
        sj.run([(c, None) for c in dprobe], [(c, None) for c in dbuild], out_cols=out_cols, out_capacity=cap)
        n = sj.last_rows
        with torch.cuda.stream(st):
            for lo in range(0, n, hq):
                m = min(hq, n - lo)
                for h, (d, _) in zip(hout, out_cols):
                    h[:m].copy_(d[lo:lo + m], non_blocking=True)
        st.synchronize()
        return n

    steps = max(1, min(args.steps, 3))
    step()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        n = step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    rows = torch.tensor([n], dtype=torch.int64, device=dev)
    dist.all_reduce(rows)
    assert int(rows.item()) == npr * world
    sj.close()
    return {"value": npr * world / dt, "unit": "rows/s", "h2d_bytes_per_step": nb * 16 + npr * 16, "d2h_bytes_per_step": int(n) * 32,
            "ms_per_step": dt * 1000.0, "steps": steps, "numa_binding": numa,
            "path": "pinned host shards -> H2D -> gsql_xchg_push of both sides -> gsql_join_* on the receive buffers -> D2H of the joined rows; "
                    "per-rank bytes; copies are not overlapped with the kernels"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
