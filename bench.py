#!/usr/bin/env python
"""bench.py - routed messages/s (send -> receive) at 1M agents, 64-way group fan-out.

Contract (driver):  python bench.py --gpus N --steps K --warmup W   (N>1 under torchrun)
prints ONE JSON line on rank 0.  `--impl reference` times the CPU restatement of the
reference path (oracle/cpu_ref.c, all host threads) on the same workload.

Workload = BASELINE config 2 (SURVEY.md section 8d "c2"): A = 1,000,000 agents, 15,625 disjoint groups
of 64 (perm = default_rng(2).permutation(A)), one step = 65,536 group sends (group ~ U, sender
~ U resampled until not a member, prio ~ U{0..3}, 256-byte [A-Za-z0-9] payloads from
default_rng(3)) = 4,194,304 routed messages, followed by a full drain of every agent
(receive_batch over all agents, max_messages = 100).

  value   device-resident: the step's sends are already staged in HBM (sdb_stage_batch); the
          timed region is submit (fan-out + commit kernels) + receive (7 kernels), timed with
          CUDA events on the launching stream, barrier + synchronize on both sides.
  e2e     the same step through the public API with HOST buffers: pinned payload/index
          arrays in, H2D inside the call, receive results copied D2H into pinned buffers.
  roofline  fan-out kernel: 280.25 algorithmic bytes per routed message (SURVEY 8d) x messages
          per launch / mean launch duration from CUDA events inside the library
          (sdb_profile), against MEASURED_PEAKS.json's copy bandwidth.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

A_AGENTS = 1_000_000
FANOUT = 64
N_GROUPS = A_AGENTS // FANOUT          # 15,625
SENDS_PER_STEP = 65_536
PAYLOAD = 256
ALG_BYTES_FANOUT = 256 + 16 + 4 + (256 + 16) / 64.0       # 280.25 B per routed message (SURVEY 8d)
ALG_BYTES_GATHER = 2 * (256 + 16)                          # gather + emit per delivered message
# Shared payloads (csrc/sdb_common.cuh; default on): a group send keeps its members' headers and ONE payload in the log,
# so the least a correct implementation must move is smaller than SURVEY's per-recipient-copy figures above:
ALG_OWN_FANOUT = 16 + 4 + (256 + 256) / 64.0               # header written + member id read + payload read/written once per send = 28 B
ALG_OWN_GATHER = (256 + 16) + 16 + 256 / 64.0              # record emitted + header read + payload read once per send = 292 B
ALNUM = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789", np.uint8)


# ------------------------------------------------------------------------------------ workload
class Workload:
    def __init__(self, n_agents=A_AGENTS, fanout=FANOUT, sends=SENDS_PER_STEP, payload=PAYLOAD):
        self.A, self.F, self.S, self.L = n_agents, fanout, sends, payload
        self.G = n_agents // fanout
        self.perm = np.random.default_rng(2).permutation(n_agents).astype(np.uint32)
        self.group_of = np.empty(n_agents, np.uint32)
        self.group_of[self.perm[: self.G * fanout]] = np.repeat(np.arange(self.G, dtype=np.uint32), fanout)
        if self.G * fanout < n_agents:
            self.group_of[self.perm[self.G * fanout:]] = 0xFFFFFFFF
        self.rng_send = np.random.default_rng(12345)
        self.rng_pay = np.random.default_rng(3)

    def members(self, g):
        return self.perm[g * self.F:(g + 1) * self.F]

    def batch(self, rng_send=None, rng_pay=None, var_len=False):
        S = self.S
        rs = rng_send if rng_send is not None else self.rng_send
        rp = rng_pay if rng_pay is not None else self.rng_pay
        grp = rs.integers(0, self.G, S).astype(np.uint32)
        snd = rs.integers(0, self.A, S).astype(np.uint32)
        while True:                                    # resample senders that are members of their group
            bad = self.group_of[snd] == grp
            nb = int(bad.sum())
            if nb == 0:
                break
            snd[bad] = rs.integers(0, self.A, nb).astype(np.uint32)
        prio = rs.integers(0, 4, S).astype(np.uint8)
        typ = np.zeros(S, np.uint8)
        lens = rs.integers(1, self.L + 1, S).astype(np.uint16) if var_len else np.full(S, self.L, np.uint16)
        off = np.arange(S, dtype=np.uint64) * self.L
        payload = ALNUM[rp.integers(0, 62, S * self.L)]
        return snd, grp, prio, typ, lens, off, payload

    # ---- verified steps (outside every timed region): batches any rank can regenerate
    PARITY_STEPS = 2

    def parity_batch(self, step, rank):
        """Step 0 has the timed shape (fixed 256-byte payloads), step 1 SURVEY 8d's correctness variant (lengths
        U[1,256]).  Seeded by (step, rank) so rank 0 can rebuild every rank's batch for the oracle."""
        seed = 7700 + 64 * step + rank
        return self.batch(np.random.default_rng(seed), np.random.default_rng(seed + 32), var_len=(step % 2 == 1))


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and clock-event (throttle) reasons through NVML every ~2 ms while the timed
    region runs (the region is only tens of milliseconds long; nvidia-smi -lms is too coarse)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, device_index=0):
        self.dev = device_index
        self.sm, self.bits, self.power = [], 0, []
        self.stop_flag = False
        self.thread = None
        self.max_mhz = None
        self.err = None

    def _run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self.dev
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.dev])
                except Exception:
                    pass
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self.stop_flag:
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                self.bits |= int(get_reasons(h))
                try:
                    self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                time.sleep(0.002)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
               "reasons": reasons, "samples": len(self.sm),
               "power_w_max": max(self.power) if self.power else None}
        if self.err:
            out["error"] = self.err
        return out


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_note(key="k_recv_gather_bytes_per_launch"):
    """DRAM bytes (read + write) per launch of a kernel from the committed ncu capture (profiles/roofline_traffic.json)."""
    p = ROOT / "profiles" / "roofline_traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(key)
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------ CPU arm
def cpu_roundtrip(wl: Workload, budget_s: float, max_batches: int):
    """Oracle port (oracle/cpu_ref.c), all host threads: fan-out + drain of c2 batches."""
    from oracle.cpu_ref import CpuOracle
    cores = os.cpu_count() or 1
    o = CpuOracle(wl.A, wl.G)
    for g in range(wl.G):
        o.create_group(g, wl.members(g))
    batches = [wl.batch() for _ in range(2)]
    o.mt_group_roundtrip(cores, *batches[0], max_messages=100)          # warm-up (page faults, allocator)
    routed = 0
    per_batch_ms = []
    t0 = time.perf_counter()
    k = 0
    while k < max_batches and (time.perf_counter() - t0) < budget_s:
        t1 = time.perf_counter()
        r, drained, _ = o.mt_group_roundtrip(cores, *batches[k % 2], max_messages=100)
        per_batch_ms.append((time.perf_counter() - t1) * 1e3)
        assert r == drained == wl.S * wl.F, (r, drained)
        routed += drained
        k += 1
    dt = time.perf_counter() - t0
    o.close()
    return routed / dt, cores, k, per_batch_ms


def oracle_parity_digests(wl: Workload, world: int, seq_base: int):
    """Ground truth for the verified steps: ONE queue (oracle/cpu_ref.c) fed every rank's parity batches in
    (step, rank) order - the order the shards import them - and drained; returns (per-agent stream digests, records).
    Uses the oracle's multi-threaded path (same streams as its single-threaded path: tests/test_oracle_c.py)."""
    from oracle.cpu_ref import CpuOracle
    cores = os.cpu_count() or 1
    o = CpuOracle(wl.A, wl.G)
    for g in range(wl.G):
        o.create_group(g, wl.members(g))
    o.digest_enable()
    o.next_seq = seq_base
    records = 0
    for step in range(wl.PARITY_STEPS):
        for r in range(world):
            routed, drained, _ = o.mt_group_roundtrip(cores, *wl.parity_batch(step, r), max_messages=1 << 30)
            assert routed == drained
            records += drained
    dg = o.digest_read()
    o.close()
    return dg, records


def parity_report(got: np.ndarray, delivered: int, wl: Workload, world: int, seq_base: int, how: str) -> dict:
    want, records = oracle_parity_digests(wl, world, seq_base)
    bad = np.nonzero(got != want)[0]
    return {"checked": True, "match": bool(len(bad) == 0 and delivered == records), "agents": int(wl.A),
            "agents_with_records": int((want != 0).sum()), "records": int(records), "records_delivered": int(delivered),
            "mismatching_agents": int(len(bad)), "steps": wl.PARITY_STEPS, "n_gpus": world,
            "stream_digest_xor": "%016x" % int(np.bitwise_xor.reduce(got)), "oracle": "oracle/cpu_ref.c (all host threads)",
            "what": "per-agent order-sensitive digest of every delivered record (32-byte header + padded payload), "
                    "include/swarmdb_b200.h 'stream digests'; " + how}


DUMP_RECORDS = 32_768            # --dump-outputs: records sampled from the step's 4,194,304 (32 MB of payload as float32)
DUMP_SEED = 2024


def dump_outputs(shard, out_dir: Path, local_rank: int, width: int) -> dict:
    """Write what the last receive delivered (still on the device after an SDB_RECV_ASYNC receive) as DIR/<name>.npy:
    every agent's record count, the step's totals, and for a fixed seeded sample of the records (`index`, positions in
    delivery order) each header field and the payload bytes (one row of `width` bytes per record, zero past its len).
    float64 where the values are integers that float32 cannot hold exactly; float32 for counts and payload bytes."""
    from cuda.bindings import runtime as cudart
    from swarmdb_b200._native import HDR_DTYPE
    total, pbytes = shard.last_receive_totals()
    cnt_dev, hdr_dev, pay_dev = shard.last_receive_dev()
    counts = np.empty(shard.stats()["n_agents"], np.uint32)
    hdr = np.empty(total, HDR_DTYPE)
    pay = np.empty(pbytes, np.uint8)
    assert cudart.cudaSetDevice(local_rank)[0] == cudart.cudaError_t.cudaSuccess
    for host, dev in ((counts, cnt_dev), (hdr, hdr_dev), (pay, pay_dev)):
        err = cudart.cudaMemcpy(host.ctypes.data, dev, host.nbytes, cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost)[0]
        assert err == cudart.cudaError_t.cudaSuccess, err
    assert int(counts.sum()) == total
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(total, min(total, DUMP_RECORDS), replace=False))
    lens = hdr["len"].astype(np.int64)
    start = np.concatenate(([0], np.cumsum((lens + 31) // 32 * 32)))[idx]        # payloads back to back, 32-byte padded
    col = np.arange(width)
    inside = col[None, :] < lens[idx][:, None]
    rows = np.where(inside, pay[np.minimum(start[:, None] + col[None, :], pbytes - 1)], 0)
    sample = hdr[idx]
    assert int(hdr["seq"].max()) < 2 ** 53                                      # exact in float64
    arrays = {"counts": counts.astype(np.float32), "totals": np.array([total, pbytes], np.float64),
              "index": idx.astype(np.float64), "payload": rows.astype(np.float32)}
    for f in HDR_DTYPE.names:
        arrays[f"header_{f}"] = sample[f].astype(np.float64)
    nbytes = sum(a.nbytes for a in arrays.values())
    assert nbytes <= 64 << 20, nbytes
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)
    return {"dir": str(out_dir), "files": sorted(f"{n}.npy" for n in arrays), "bytes": nbytes, "records": total,
            "records_sampled": len(idx)}


WORKLOAD_C2 = ("c2: 1M agents, 15625 groups x 64, 65536 group sends/step (4,194,304 routed msgs), "
               "256-byte payloads, full drain (receive_batch all agents, max_messages=100) each step")


def workload_c3(world: int) -> str:
    return (f"c3: c2's workload (1M agents, 15625 groups x 64, 256-byte payloads) with agents hash-sharded "
            f"(fnv1a64 % {world}) over {world} GPUs; every rank ingests 65536 group sends/step; each shard drains its agents")


def reference_python_leg(budget_s: float):
    """BASELINE.md section 3 'reference-python': the reference's own class (staged by oracle/build_ref.py) over the
    in-memory broker stub, one core: c1 exactly + a reduced c2.  None when the reference file is not available."""
    if budget_s <= 0:
        return None
    try:
        from oracle import ref_bench
        return ref_bench.run_all(budget_s)
    except Exception as e:  # pragma: no cover  (reported, never fatal for the GPU line)
        return {"kind": "reference", "unavailable": repr(e)}


def run_reference(args, rank, world):
    """Reference arm: the CPU restatement of the path (oracle/cpu_ref.c, all host threads) on the arm's own
    workload, `--warmup` untimed batches then `--steps` timed ones; the reference's own Python class is timed
    beside it on a bounded sample (`cpu_baseline_reference`)."""
    if rank != 0:
        return
    from oracle.cpu_ref import CpuOracle
    wl = Workload()
    cores = os.cpu_count() or 1
    o = CpuOracle(wl.A, wl.G)
    for g in range(wl.G):
        o.create_group(g, wl.members(g))
    batches = [wl.batch() for _ in range(2)]
    for i in range(max(args.warmup, 1)):                                  # untimed: page faults, allocator, thread start
        o.mt_group_roundtrip(cores, *batches[i % 2], max_messages=100)
    per, routed = [], 0
    t0 = time.perf_counter()
    k = 0
    while k < args.steps:
        t1 = time.perf_counter()
        r, drained, _ = o.mt_group_roundtrip(cores, *batches[k % 2], max_messages=100)
        per.append((time.perf_counter() - t1) * 1e3)
        assert r == drained == wl.S * wl.F, (r, drained)
        routed += drained; k += 1
    value = routed / (time.perf_counter() - t0)
    o.close()
    sample = (f"{k} full c2 batch(es) of {wl.S} group sends x {wl.F} (= {wl.S * wl.F} routed msgs each): route + "
              f"materialise + drain, {cores} threads, each inbox written by one thread")
    line = {
        "impl": "reference", "metric": "messages/sec routed (send->receive) at 1M agents, 64-way fanout",
        "value": value, "unit": "messages/s", "n_gpus": args.gpus, "steps": k, "warmup": max(args.warmup, 1),
        "ms_per_step": float(np.mean(per)) if per else None, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_C2 if args.gpus == 1 else workload_c3(args.gpus),
                   "impl_detail": "CPU restatement of the reference path (oracle/cpu_ref.c, pinned to goldens produced by "
                                  "the unmodified reference); one host, all threads; at --gpus N the CPU arm still runs "
                                  "one c2 batch per step on this host"},
        "cpu_baseline": {"value": value, "unit": "messages/s", "cores": cores, "kind": "port", "sample": sample},
        "cpu_baseline_reference": reference_python_leg(args.ref_budget),
        "e2e": {"value": value, "unit": "messages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ the other BASELINE configs
def config_c1(tmp="/tmp/sdb_bench_c1"):
    """BASELINE config 1 through the drop-in Python surface: 2 agents, 1,000 point-to-point 128-byte messages
    (content from default_rng(1)), then agent_b drains.  Check: delivered contents == sent contents, in order."""
    import swarmdb_b200 as sdb
    rng = np.random.default_rng(1)
    contents = [ALNUM[rng.integers(0, 62, 128)].tobytes().decode() for _ in range(1000)]
    db = sdb.SwarmsDB(save_dir=tmp, auto_save=False,
                      gpu_config=sdb.GpuConfig(max_agents=1024, ring_slots=2048, arena_bytes=1 << 26))
    db.register_agent("agent_a"); db.register_agent("agent_b")
    for c in contents[:50]:                                   # warm-up (allocator, first launches)
        db.send_message("agent_a", c, "agent_b")
    db.receive_messages("agent_b", 100)
    clocks = ClockSampler(0); clocks.start()
    t0 = time.perf_counter()
    for c in contents:
        db.send_message("agent_a", c, "agent_b")
    t1 = time.perf_counter()
    got = db.receive_messages("agent_b", 2000)
    t2 = time.perf_counter()
    clk = clocks.stop()
    ok = [m.content for m in got] == contents and all(m.sender_id == "agent_a" for m in got)
    db.close()
    return {"config": "c1: 2 agents, 1k point-to-point 128-byte messages through swarmdb_b200.SwarmsDB (buffered sends, "
                      "one flush at receive)", "unit": "messages/s",
            "send_msgs_per_s": 1000 / (t1 - t0), "receive_msgs_per_s": 1000 / (t2 - t1), "value": 1000 / (t2 - t0),
            "check": {"what": "delivered contents and order == sent (M:553-601)", "ok": bool(ok)}, "clocks": clk}


def config_c4(sweeps=4):
    """BASELINE config 4: 10,048 agents (157 groups x 64) x 10,000 pending 256-byte records each, 4 priority levels;
    receive_batch(all agents, max_messages=100, PRIORITY).  Check: the per-agent stream digests of 8 sampled groups
    (512 agents) after the timed sweeps against oracle/cpu_ref.c fed the same sends with the same sequence numbers."""
    from oracle.cpu_ref import CpuOracle
    from swarmdb_b200._native import RECV_PRIORITY, Shard
    peak, src = hbm_peak()
    G, F, depth, L = 157, 64, 10_000, 256
    A = G * F
    S = 65536
    shard = Shard(max_agents=A, ring_slots=16384, arena_bytes=1 << 35, max_payload_bytes=L, max_groups=G,
                  max_batch_sends=S, max_batch_payload=S * L, max_recv_records=A * 100 + 4096,
                  max_recv_payload=(A * 100 + 4096) * L)
    rng = np.random.default_rng(4)
    perm = rng.permutation(A).astype(np.uint32)
    group_of = np.empty(A, np.uint32); group_of[perm] = np.repeat(np.arange(G, dtype=np.uint32), F)
    sample_groups = np.sort(rng.choice(G, 8, replace=False)).astype(np.uint32)
    in_sample = np.zeros(G, bool); in_sample[sample_groups] = True
    sample_agents = np.sort(np.concatenate([perm[g * F:(g + 1) * F] for g in sample_groups])).astype(np.uint32)
    cpu = CpuOracle(A, G)
    for g in range(G):
        shard.create_group(g, perm[g * F:(g + 1) * F])
        if in_sample[g]:
            cpu.create_group(g, perm[g * F:(g + 1) * F])
    cpu.digest_enable(); shard.digest_reset()
    total_sends = G * depth
    grp_all = np.repeat(np.arange(G, dtype=np.uint32), depth)
    rng.shuffle(grp_all)
    t0 = time.perf_counter()
    for s0 in range(0, total_sends, S):
        grp = grp_all[s0:s0 + S]
        n = len(grp)
        snd = rng.integers(0, A, n).astype(np.uint32)
        bad = group_of[snd] == grp
        while bad.any():                                      # sender outside its group: every member gets the record
            snd[bad] = rng.integers(0, A, int(bad.sum())).astype(np.uint32)
            bad = group_of[snd] == grp
        prio = rng.integers(0, 4, n).astype(np.uint8)
        lens = np.full(n, L, np.uint16)
        off = np.arange(n, dtype=np.uint64) * L
        pay = ALNUM[rng.integers(0, 62, n * L)]
        base = shard.send_group_batch(snd, grp, prio, None, lens, off, pay)
        keep = in_sample[grp]
        if keep.any():                                        # the oracle sees only the sampled groups, same sequence numbers
            idx = np.nonzero(keep)[0]
            seq0 = (base + idx.astype(np.uint64) * F).astype(np.uint64)
            cpu.send_group_seq(snd[idx], grp[idx], prio[idx], np.zeros(len(idx), np.uint8), lens[idx], off[idx], pay, seq0)
    shard.sync()
    load_s = time.perf_counter() - t0
    st = shard.stats()
    assert st["enqueued"] == A * depth and st["ring_overflow"] == 0, st
    shard.profile(True)
    clocks = ClockSampler(0); clocks.start()
    wall = []
    for _ in range(sweeps):
        t1 = time.perf_counter()
        _, total, _ = shard.receive_batch(None, 100, RECV_PRIORITY, copy_out=False)
        wall.append((time.perf_counter() - t1) * 1e3)
        assert total == A * 100
        shard.digest_fold()
    clk = clocks.stop()
    prof = shard.profile_read()
    for _ in range(sweeps):
        cpu.receive_counts(sample_agents, 100, RECV_PRIORITY)
    ok = bool(np.array_equal(shard.digest_read(sample_agents), cpu.digest_read(sample_agents)))
    shard.close(); cpu.close()
    k5_ms = sum(v[0] for k, v in prof.items() if k.startswith("recv")) / sweeps
    alg = A * (depth * 1 + 2 * 100 * (L + 16))               # SURVEY 8d: 64,400 B per agent-call
    return {"config": f"c4: {A} agents x {depth} pending {L}-byte records, 4 priorities, receive_batch(all, 100, PRIORITY)",
            "preload_s": load_s, "sweep_wall_ms": wall, "p50_sweep_wall_ms": float(np.median(wall)),
            "k5_kernels_ms_per_sweep": k5_ms,
            "kernels_ms": {k: v[0] / v[1] for k, v in prof.items() if v[1]},
            "per_agent_call_us": k5_ms * 1e3 / A, "value": A * 100 / (k5_ms * 1e-3), "unit": "messages/s dequeued",
            "roofline": {"bound": "hbm", "algorithmic_bytes_per_sweep": alg, "achieved": alg / (k5_ms * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": alg / (k5_ms * 1e-3) / 1e9 / peak, "peak_source": src},
            "check": {"what": f"stream digests of {len(sample_agents)} agents (8 sampled groups) after {sweeps} priority sweeps "
                              "== oracle/cpu_ref.c (priority desc, arrival asc; App. A rule 9)", "ok": ok},
            "clocks": clk}


def config_c5(n_req=1_000_000, n_backends=256):
    """BASELINE config 5: 1M unit-cost requests over 256 backends, weights U{1..8}; both pick modes, bit-exact against
    the oracle's sequential definition (include/swarmdb_b200.h)."""
    from oracle.cpu_ref import CpuOracle
    from swarmdb_b200._native import Shard
    rng = np.random.default_rng(5)
    w = rng.integers(1, 9, n_backends)
    out = {"config": f"c5: {n_req} unit-cost requests over {n_backends} backends, weights U{{1..8}}, load0 = 0",
           "unit": "picks/s", "note": "not HBM-bound: the 256-entry table lives in shared memory / L1 (SURVEY 8d)"}
    clocks = ClockSampler(0); clocks.start()
    ok = True
    for mode, name in ((0, "weighted_least_load"), (1, "weighted_random")):
        g = Shard(max_agents=16)
        g.set_backends(w)
        g.select_backends(1000, None, mode, 6)                   # warm-up
        g.set_backends(w)
        t0 = time.perf_counter()
        picks = g.select_backends(n_req, None, mode, 6)
        wall = time.perf_counter() - t0
        o = CpuOracle(16)
        o.set_backends(w)
        t1 = time.perf_counter()
        ref = o.select_backends(n_req, None, mode, 6)
        cpu_s = time.perf_counter() - t1
        same = bool(np.array_equal(picks, ref) and np.array_equal(g.backend_loads(), o.backend_loads()))
        ok = ok and same
        out[name] = {"picks_per_s_end_to_end": n_req / wall, "wall_ms": wall * 1e3,
                     "cpu_oracle_picks_per_s_1_core": n_req / cpu_s, "bit_exact_vs_oracle": same}
        g.close(); o.close()
    out["clocks"] = clocks.stop()
    out["value"] = out["weighted_least_load"]["picks_per_s_end_to_end"]
    out["check"] = {"what": "picks and final loads == oracle (sequential greedy / exponential race)", "ok": ok}
    return out


# ------------------------------------------------------------------------------------ GPU arm
def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - swarmdb_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL prints its version banner to stdout at communicator creation: keep stdout to the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    from swarmdb_b200._native import Shard

    wl = Workload()
    if world > 1:
        from swarmdb_b200.sharded import run_sharded_bench
        return run_sharded_bench(args, rank, world, local_rank, wl)

    stream = torch.cuda.Stream()
    K, W = args.steps, args.warmup
    ring_slots = int(os.environ.get("SDB_RING_SLOTS", "64"))
    shard = Shard(max_agents=wl.A, ring_slots=ring_slots, arena_bytes=1 << 33, max_payload_bytes=wl.L, max_groups=1 << 14,
                  member_pool_entries=wl.A + 1024, max_batch_sends=wl.S, max_batch_payload=wl.S * wl.L,
                  max_recv_records=wl.S * wl.F + (1 << 16), max_recv_payload=(wl.S * wl.F + (1 << 16)) * wl.L,
                  device=local_rank, fanout_variant=args.variant)
    shard.set_stream(stream.cuda_stream)
    shard.register(np.arange(wl.A, dtype=np.uint32))
    for g in range(wl.G):
        shard.create_group(g, wl.members(g))
    shard.sync()

    n_distinct = min(W + K, 8)
    host_batches = [wl.batch() for _ in range(n_distinct)]
    staged = [shard.stage(1, *b) for b in host_batches]
    per_step_msgs = wl.S * wl.F

    def device_step(i):
        # device-resident step: fan-out + index build + full drain are only ENQUEUED (SDB_RECV_ASYNC); the records a
        # step delivered are read back from the device counters after the timed region, not step by step
        shard.submit(staged[i % n_distinct])
        shard.receive_batch(None, 100, 0, copy_out=False, wait=False)

    with torch.cuda.stream(stream):
        for i in range(W):
            device_step(i)
            assert shard.last_receive_totals()[0] == per_step_msgs
        st0 = shard.stats()
        launches0 = st0["kernel_launches"]
        shard.profile(True)
        clocks = ClockSampler(local_rank); clocks.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(stream)
        for i in range(K):
            device_step(W + i)
        ev1.record(stream)
        torch.cuda.synchronize()
        clk = clocks.stop()
        ms_total = ev0.elapsed_time(ev1)
        prof = shard.profile_read()
        shard.profile(False)
        st1 = shard.stats()
        launches = st1["kernel_launches"] - launches0
        delivered = st1["delivered"] - st0["delivered"]          # counted on the device by the receive kernels
        assert st1["ring_overflow"] == 0 and shard.last_receive_totals()[0] == per_step_msgs
        if args.dump_outputs:                              # untimed; before the sustained block reuses the receive buffers
            info = dump_outputs(shard, Path(args.dump_outputs), local_rank, wl.L)
            print(f"bench.py: step {W + K - 1} outputs written: {json.dumps(info)}", file=sys.stderr, flush=True)
        # sustained figure: the same step repeated for a few hundred milliseconds (clocks and power settle), timed as one block
        sustained = None
        if args.sustained_steps > 0:
            Ks = args.sustained_steps
            clocks_s = ClockSampler(local_rank); clocks_s.start()
            torch.cuda.synchronize()
            ev0.record(stream)
            for i in range(Ks):
                device_step(W + K + i)
            ev1.record(stream)
            torch.cuda.synchronize()
            ms_s = ev0.elapsed_time(ev1)
            st2 = shard.stats()
            assert st2["delivered"] - st1["delivered"] == Ks * per_step_msgs and st2["ring_overflow"] == 0
            sustained = {"steps": Ks, "ms_per_step": ms_s / Ks, "value": Ks * per_step_msgs / (ms_s * 1e-3), "unit": "messages/s",
                         "clocks": clocks_s.stop()}
    assert delivered == K * per_step_msgs, (delivered, K * per_step_msgs)
    value = delivered / (ms_total * 1e-3)

    if args.no_extras:
        print(json.dumps({"value": value, "ms_per_step": ms_total / K, "steps": K, "clocks": clk,
                          "kernels": {k: (v[0] / v[1] if v[1] else None) for k, v in prof.items() if v[1]}}), flush=True)
        return
    # ---- e2e: host buffers through the public bulk API, H2D and D2H inside the timed region
    rec_cap = per_step_msgs + (1 << 16)
    from swarmdb_b200._native import HDR_DTYPE
    pin_hdr = torch.empty(rec_cap * 32, dtype=torch.uint8, pin_memory=True).numpy().view(HDR_DTYPE)
    pin_pay = torch.empty(rec_cap * wl.L, dtype=torch.uint8, pin_memory=True).numpy()
    pinned_in = []
    for b in host_batches[: min(n_distinct, 4)]:
        t = torch.empty(b[6].nbytes, dtype=torch.uint8, pin_memory=True)
        t.numpy()[:] = b[6]
        pinned_in.append(b[:6] + (t.numpy(),))
    Ke = max(1, min(K, 8))

    def e2e_step(i):
        b = pinned_in[i % len(pinned_in)]
        shard.send_group_batch(*b)
        cnt, hdr, pay = shard.receive_batch(None, 100, 0, copy_out=True, out_hdr=pin_hdr, out_payload=pin_pay)
        return len(hdr), int(hdr["seq"][-1]) if len(hdr) else 0

    with torch.cuda.stream(stream):
        for i in range(2):
            assert e2e_step(i)[0] == per_step_msgs
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        e0.record(stream)
        got = 0
        for i in range(Ke):
            got += e2e_step(i)[0]
        e1.record(stream)
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t_wall) * 1e3
        e2e_ms = max(e0.elapsed_time(e1), wall_ms)          # host-side work between calls counts too
    e2e_value = got / (e2e_ms * 1e-3)
    h2d = wl.S * wl.L + wl.S * 64                            # payload + 64-byte descriptors built by the library
    d2h = per_step_msgs * (32 + wl.L) + wl.A * 4 + 16        # headers + payloads + per-agent counts + totals

    # ---- p50 dequeue: one receive_batch([agent], max_messages=100) through ctypes -> kernels -> D2H,
    # host buffers, >= 1 message pending (SURVEY 8d); 2000 distinct agents after one more group batch
    shard.send_group_batch(*pinned_in[0])
    shard.sync()
    probe = np.random.default_rng(99).permutation(wl.A)[:2200].astype(np.uint32)
    lat = []
    lat_launch = []
    clocks_p50 = ClockSampler(local_rank); clocks_p50.start()
    for k, a in enumerate(probe[:1100]):                       # the launched path: kernel + D2H + stream sync per call
        ai = int(a)
        t1 = time.perf_counter()
        h, _, _ = shard.receive_one(ai, 100, 0)
        dt = time.perf_counter() - t1
        if k >= 100 and len(h):
            lat_launch.append(dt * 1e6)
    shard.latency_server(True)                                 # the persistent dequeue server: mailbox in pinned memory
    for k, a in enumerate(probe[1100:]):
        ai = int(a)
        t1 = time.perf_counter()
        h, _, _ = shard.receive_one(ai, 100, 0)
        dt = time.perf_counter() - t1
        if k >= 100 and len(h):
            lat.append(dt * 1e6)
    shard.latency_server(False)
    clk_p50 = clocks_p50.stop()
    p50 = float(np.percentile(lat, 50)) if lat else None
    p99 = float(np.percentile(lat, 99)) if lat else None
    shard.receive_batch(None, 100, 0, copy_out=False)          # drain the rest

    # ---- content parity at the benchmarked size (outside every timed region): two verified steps through the same
    # calls, every agent's stream digested on the device, against one oracle queue fed the same batches
    while shard.receive_batch(None, 100, 0, copy_out=False)[1]:
        pass
    shard.digest_reset()
    seq_base = shard.stats()["next_seq"]
    p_delivered = 0
    for step in range(wl.PARITY_STEPS):
        shard.send_group_batch(*wl.parity_batch(step, 0))
        _, t, _ = shard.receive_batch(None, 100, 0, copy_out=False)
        shard.digest_fold()
        p_delivered += t
    while True:
        _, t, _ = shard.receive_batch(None, 100, 0, copy_out=False)
        shard.digest_fold()
        if t == 0:
            break
        p_delivered += t
    parity = parity_report(shard.digest_read(), p_delivered, wl, 1, seq_base,
                           "sdb_send_group_batch + sdb_receive_batch on one GPU")

    # ---- roofline: the DOMINANT kernel of the step is the receive gather; the fan-out (north_star's 60 % target) and the
    # whole step (825 B per routed message, SURVEY 8d) are reported beside it
    peak, peak_src = hbm_peak()
    fan_ms, fan_n = prof["fanout"]
    fan_avg_ms = fan_ms / max(fan_n, 1)
    gat_ms, gat_n = prof["recv_gather"]
    gat_avg = gat_ms / max(gat_n, 1)
    achieved = ALG_BYTES_GATHER * per_step_msgs / (gat_avg * 1e-3) / 1e9 if gat_n else 0.0
    kernels = {k: {"ms_per_launch": (v[0] / v[1] if v[1] else None), "launches": v[1]} for k, v in prof.items() if v[1]}
    kernels["fanout"]["achieved_gbs"] = ALG_BYTES_FANOUT * per_step_msgs / (fan_avg_ms * 1e-3) / 1e9 if fan_n else None
    kernels["fanout"]["frac"] = kernels["fanout"]["achieved_gbs"] / peak if fan_n else None
    kernels["fanout"]["algorithmic_bytes_per_msg"] = ALG_BYTES_FANOUT
    kernels["fanout"]["traffic"] = traffic_note("k_group_fanout_bytes_per_launch")
    step_alg = (ALG_BYTES_FANOUT + 1 + ALG_BYTES_GATHER) * per_step_msgs        # 825.25 B per routed message
    from swarmdb_b200._native import shared_payload_enabled
    shared_payloads = shared_payload_enabled()
    own = None
    if shared_payloads:
        kernels["fanout"]["own_layout"] = {"algorithmic_bytes_per_msg": ALG_OWN_FANOUT,
                                           "frac": ALG_OWN_FANOUT * per_step_msgs / (fan_avg_ms * 1e-3) / 1e9 / peak if fan_n else None}
        own = {"what": "shared payloads: the log keeps one payload per group send, not one per recipient, so the step moves fewer "
                       "bytes than SURVEY 8(d)'s per-recipient-copy figures (kept as `achieved` / `frac` / `step_frac` so that rounds "
                       "stay comparable; they can exceed what DRAM could deliver for that algorithm). Against the least this "
                       "layout must move:",
               "gather_bytes_per_msg": ALG_OWN_GATHER, "gather_frac": ALG_OWN_GATHER * per_step_msgs / (gat_avg * 1e-3) / 1e9 / peak if gat_n else None,
               "step_bytes_per_msg": ALG_OWN_FANOUT + 1 + ALG_OWN_GATHER,
               "step_frac": (ALG_OWN_FANOUT + 1 + ALG_OWN_GATHER) * per_step_msgs / ((ms_total / K) * 1e-3) / 1e9 / peak}

    # ---- CPU baseline beside it (rank 0, N=1): bounded sample of the same workload
    if args.cpu_budget > 0:
        cpu_value, cores, kb, _ = cpu_roundtrip(wl, budget_s=args.cpu_budget, max_batches=8)
    else:
        cpu_value, cores, kb = None, os.cpu_count(), 0

    line = {
        "metric": "messages/sec routed (send->receive) at 1M agents, 64-way fanout",
        "value": value, "unit": "messages/s", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_C2,
                   "l2": "inputs larger than L2: each step writes 1.2 GB of records into an 8 GiB arena and reads "
                         "them back; no explicit flush needed",
                   "fanout_variant": args.variant, "ring_slots": ring_slots, "arena_bytes": 1 << 33,
                   "shared_payloads": shared_payloads},
        "clocks": clk,
        "sustained": sustained,
        "e2e": {"value": e2e_value, "unit": "messages/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": Ke, "ms_per_step": e2e_ms / Ke},
        "gpu_launches": int(launches),
        "p50_dequeue_us": p50, "p99_dequeue_us": p99,
        "parity": parity,
        "roofline": {"kernel": "k_recv_gather_tma (dominant: %.0f %% of the step)" % (100 * gat_avg / (ms_total / K)),
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic_note(), "peak_source": peak_src,
                     "algorithmic_bytes_per_msg": ALG_BYTES_GATHER, "msgs_per_launch": per_step_msgs,
                     "ms_per_launch": gat_avg,
                     "step_frac": step_alg / ((ms_total / K) * 1e-3) / 1e9 / peak,
                     "step_algorithmic_bytes_per_msg": ALG_BYTES_FANOUT + 1 + ALG_BYTES_GATHER,
                     "own_layout": own},
        "kernels": kernels,
        "cpu_baseline": {"value": cpu_value, "unit": "messages/s", "cores": cores, "kind": "port",
                         "sample": f"{kb} full c2 batch(es) (4,194,304 routed msgs each), route + materialise + drain, "
                                   f"oracle/cpu_ref.c on {cores} threads"},
        "cpu_baseline_reference": reference_python_leg(args.ref_budget),
    }
    for s in staged:
        shard.free_staged(s)
    shard.close()
    # ---- the other BASELINE configs, each with its own clock record and oracle check (the c2 shard is gone: c4 alone
    # keeps 29 GB of records in HBM)
    configs = {"c2": {"see": "top level of this line"},
               "p50_dequeue": {"config": "one receive_batch([agent], max_messages=100) through ctypes -> kernel -> D2H with >= 1 "
                                         "message pending, 2000 agents of the c2 queue", "p50_us": p50, "p99_us": p99,
                               "path": "persistent dequeue server (sdb_latency_server): request in mapped pinned memory, answer "
                                       "written by the kernel into pinned host memory",
                               "launched_path_p50_us": float(np.percentile(lat_launch, 50)) if lat_launch else None,
                               "clocks": clk_p50, "check": {"what": "every probe returned its pending records", "ok": bool(lat)}}}
    if not args.skip_configs:
        for name, fn in (("c1", config_c1), ("c4", config_c4), ("c5", config_c5)):
            try:
                configs[name] = fn()
            except Exception as e:  # pragma: no cover  (reported in the line, never fatal for c2)
                configs[name] = {"error": repr(e)}
    line["configs"] = configs
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", type=int, default=int(os.environ.get("SDB_FANOUT_VARIANT", "2")))
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--ref-budget", type=float, default=20.0,
                    help="seconds for the reference-python leg (the reference's own class on one core); 0 = skip")
    ap.add_argument("--skip-configs", action="store_true", help="skip the c1 / c4 / c5 legs of the N=1 line")
    ap.add_argument("--sustained-steps", type=int, default=300,
                    help="extra block of steps after the K timed ones, timed as a whole and reported under `sustained` (0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="profiling runs: only the device-resident timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one delivered (per-agent counts, a seeded sample of "
                         "the records' headers and payloads) as DIR/<name>.npy; one GPU only")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or world != 1):
        ap.error("--dump-outputs needs the GPU arm on one GPU (--impl ours, no torchrun)")
    if args.warmup < 3:
        args.warmup = 3
    if args.no_extras:
        args.sustained_steps = 0
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
