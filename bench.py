#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its configs[1]: 4 KiB random-read IOPS on one 8 GiB
HBM-resident Malloc bdev per GPU (qd=32 per request queue, Q queues), plus 128 KiB sequential GB/s.

  python bench.py [--gpus N --steps K --warmup W]            our CUDA path  (one rank per GPU under torchrun)
  python bench.py --impl reference [...]                      the reference's CPU path on the host cores

One "step" = one pass of the hot path over one batch: every queue of the LUN gets `per_queue`
requests and the LUN is kicked once.  `value` is measured with requests, SG lists, client buffers
and completions resident in HBM (CUDA events on the LUN's stream); `e2e` goes through the C ABI
with host arrays and pinned host client buffers, PCIe traffic inside the timed region.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from oim_b200 import abi, traces  # noqa: E402

NUM_BLOCKS = 16777216          # 8 GiB / 512 B  (BASELINE.json configs[1])
BLOCK = 512


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # 254 request queues = the most a vhost-scsi controller can have (256 virtqueues minus control and event queue,
    # S/lib/vhost/vhost_internal.h:63, rte_vhost/vhost.h:130) x 16512 requests ~ the 2^22-request C2 trace of SURVEY.md 8(d)
    p.add_argument("--queues", type=int, default=int(os.environ.get("OIM_BENCH_QUEUES", 254)))
    p.add_argument("--per-queue", type=int, default=int(os.environ.get("OIM_BENCH_PER_QUEUE", 16512)))
    p.add_argument("--seq-queues", type=int, default=256)
    p.add_argument("--seq-per-queue", type=int, default=256)
    p.add_argument("--e2e-queues", type=int, default=256)
    p.add_argument("--e2e-per-queue", type=int, default=512)
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--ref-procs", type=int, default=0, help="reference reactors (processes) of --impl reference; 0 = one per LUN of the job (= --gpus); capped by cores, memory budget and 8")
    p.add_argument("--no-seq", action="store_true", help="skip the 128 KiB sequential leg")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-vq", action="store_true", help="skip the virtqueue-mode leg")
    p.add_argument("--no-mixed", action="store_true", help="skip the 70/30 mixed leg (config 4 shape)")
    p.add_argument("--no-lat", action="store_true", help="skip the single-queue qd=32 closed-loop leg")
    p.add_argument("--no-vu", action="store_true", help="skip the leg through the daemon's vhost-user socket")
    p.add_argument("--no-poller-leg", action="store_true", help="skip the resident-poller-in-HBM leg")
    p.add_argument("--no-numa", action="store_true", help="do not bind the rank to the GPU's NUMA node")
    p.add_argument("--no-sweep", action="store_true", help="skip the queue-count sweep (1..1024 request queues)")
    p.add_argument("--no-mirror", action="store_true", help="skip the mirrored-bdev leg (config 5; runs when --gpus >= 2)")
    p.add_argument("--no-extra", action="store_true", help="skip the 4 KiB random-write / 128 KiB sequential-read legs")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps of the headline leg, write what its last step returned (completion fields "
                        "and read payload of a fixed sample of requests) as DIR/<name>.npy, for comparing two builds")
    return p.parse_args()


DUMP_REQUESTS = 2048           # 2048 x 4 KiB of payload as float32 = 32 MiB


def dump_outputs(out_dir: str, prefix: str, t: traces.Trace, arena, cpls: np.ndarray, torch) -> None:
    """What a caller of a single-element-SG leg receives after its last step, for a fixed, seeded sample of its requests:
    the completion fields the reference defines plus data_transferred, and each request's client buffer (`arena`, a
    CUDA tensor).  Values are exact in float64 (completion fields) and float32 (bytes)."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(t.reqs)
    assert len(t.iovs) == n, "one SG element per request"
    idx = np.sort(np.random.default_rng(0xD0).choice(n, size=min(n, DUMP_REQUESTS), replace=False))
    buf = t.iovs[idx]
    ln = int(buf["len"][0])
    assert (buf["len"] == ln).all()
    off = torch.from_numpy(buf["addr"].astype(np.int64)).to(arena.device)
    payload = arena[off[:, None] + torch.arange(ln, device=arena.device)[None, :]].cpu().numpy()
    np.save(os.path.join(out_dir, f"{prefix}_request_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, f"{prefix}_payload.npy"), payload.astype(np.float32))
    for f in abi.CPL_PARITY_FIELDS + ("data_transferred",):
        np.save(os.path.join(out_dir, f"{prefix}_cpl_{f}.npy"), cpls[f][idx].astype(np.float64))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(key: str, requests_per_launch: int):
    """DRAM bytes per launch from the committed ncu capture, scaled if the launch size differs"""
    try:
        e = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[key]
        return e["dram_bytes_per_launch"] * requests_per_launch / e["requests_per_launch"]
    except (OSError, KeyError, ValueError):
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "25"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def shard_plan(rank: int, world: int) -> dict:
    """SURVEY.md 8(e): LUNs are independent units; LUN i (its bdev, controller, trace seed) lives on
    rank i = GPU i.  No state is shared between ranks, so there is no data-path collective."""
    assert 0 <= rank < world
    return {"bdev": f"Malloc{rank}", "ctrlr": f"vhost.{rank}", "target": 0, "store_seed": 0xB2000000 + rank,
            "trace_seed": 0xB2000000 + rank, "e2e_seed": 0xE2E00000 + rank}


def aggregate(units_per_rank: int, steps: int, world: int, max_ms: float) -> float:
    """whole-job throughput: units processed by ALL ranks / the slowest rank's device time"""
    return units_per_rank * steps * world / (max_ms / 1e3)


def dist_setup(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own C on the host cores
# ------------------------------------------------------------------------------------------------

class CpuLeg:
    """Replay the workload through oracle/_ref (the compiled reference) or, where that did not
    travel, the C restatement.  One thread: SPDK polls one vhost controller - hence one LUN - on
    one reactor core (S/lib/vhost/vhost_scsi.c:1314-1318)."""

    def __init__(self, io_blocks: int = 8, pattern: str = "randread"):
        from oracle import bindings
        try:
            bindings.build()
        except Exception:  # noqa: BLE001  (prebuilt libraries may be all there is on the GPU box)
            pass
        cls, self.kind = ((bindings.RefOracle, "reference") if bindings.ref_available()
                          else (bindings.PortOracle, "port"))
        self.o = cls(NUM_BLOCKS, BLOCK)
        self.io_bytes, self.pattern = io_blocks * BLOCK, pattern
        self.chunk = (1 << 18) if io_blocks <= 8 else (1 << 13)
        self.t = traces.uniform_trace(self.chunk, NUM_BLOCKS, io_blocks=io_blocks, pattern=pattern, seed=0xB2000000)
        self.arena = np.zeros(self.t.arena_bytes, dtype=np.uint8)
        if "write" in pattern:
            self.arena[:] = traces.pattern_bytes(0xC3, 0, self.arena.size)
        self.iovs = self.t.bind(self.arena.ctypes.data)
        self.o.submit(self.t.reqs[:4096], self.iovs)                       # warm-up pass

    def run(self, seconds: float):
        """-> (iops, info): IOPS over the time spent inside the reference's poller
        (process_requestq + completion polling), not this harness's descriptor building"""
        done, t0, wall = 0, time.perf_counter(), 0.0
        self.o.busy_ns(reset=True)
        while time.perf_counter() - t0 < seconds:
            a = time.perf_counter()
            self.o.submit(self.t.reqs, self.iovs)
            wall += time.perf_counter() - a
            done += self.chunk
        busy = self.o.busy_ns(reset=True) / 1e9 or wall
        return done / busy, {
            "kind": self.kind, "cores": 1, "unit": "IOPS",
            "sample": f"{done} x {self.io_bytes} B {self.pattern} requests over the 8 GiB bdev, {busy:.1f} s inside the "
                      f"reference's poller ({wall:.1f} s incl. the harness building vring descriptors); "
                      f"{self.chunk}-request trace replayed; client buffers {self.arena.size >> 20} MiB host memory; "
                      f"1 reactor thread (SPDK: one core per vhost controller)"}

    def close(self):
        self.o.close()


def _cpu_worker(conn, io_blocks: int, pattern: str):
    """one reference reactor: its own process, its own controller + 8 GiB Malloc bdev, its own trace"""
    try:
        leg = CpuLeg(io_blocks, pattern)
        conn.send(("ready", leg.kind))
        while True:
            msg = conn.recv()
            if msg[0] == "run":
                v, info = leg.run(msg[1])
                conn.send(("done", v, info))
            else:
                break
        leg.close()
    except Exception as e:  # noqa: BLE001
        conn.send(("error", f"{type(e).__name__}: {e}"))


def host_memory_budget() -> int:
    """bytes this process tree may safely take: the smaller of MemAvailable and the cgroup limit (a container's
    /proc/meminfo shows the HOST's memory; exceeding the cgroup limit takes the whole box down), quartered"""
    avail = 1 << 62
    for ln in open("/proc/meminfo"):
        if ln.startswith("MemAvailable:"):
            avail = int(ln.split()[1]) * 1024
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(path).read().strip()
            if v.isdigit():
                avail = min(avail, int(v))
        except OSError:
            pass
    return avail // 4


def cpu_reactor_count(want: int) -> int:
    """how many reference reactors can run side by side: every reactor is a process with its own 8 GiB bdev and
    1 GiB of client buffers; never more than the usable cores, the memory budget, or 8"""
    cores = len(os.sched_getaffinity(0))
    by_mem = int(host_memory_budget() // ((NUM_BLOCKS * BLOCK) + (3 << 29)))
    return max(1, min(want, cores, by_mem, 8))


class CpuFarm:
    """the reference on all the host cores it can use: P independent reactors, as `vhost -m <mask>` with one
    controller per core would run them; the aggregate is the sum of their rates over the same wall interval"""

    def __init__(self, nproc: int, io_blocks: int = 8, pattern: str = "randread"):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.workers = []
        for _ in range(nproc):
            parent, child = ctx.Pipe()
            pr = ctx.Process(target=_cpu_worker, args=(child, io_blocks, pattern), daemon=True)
            pr.start()
            self.workers.append((pr, parent))
        self.kind = None
        for _, c in self.workers:
            msg = c.recv()
            if msg[0] != "ready":
                raise RuntimeError(f"reference reactor failed to start: {msg}")
            self.kind = msg[1]

    def run(self, seconds: float):
        for _, c in self.workers:
            c.send(("run", seconds))
        vals, info = [], None
        for _, c in self.workers:
            msg = c.recv()
            if msg[0] != "done":
                raise RuntimeError(f"reference reactor failed: {msg}")
            vals.append(msg[1])
            info = msg[2]
        return vals, info

    def close(self):
        for pr, c in self.workers:
            try:
                c.send(("close",))
            except Exception:  # noqa: BLE001
                pass
        for pr, _ in self.workers:
            pr.join(20)
            if pr.is_alive():
                pr.kill()


def run_reference(args, rank, world):
    if rank != 0:
        return
    per_step = max(0.5, min(20.0, 100.0 / max(1, args.steps + args.warmup)))
    # The configuration decides how many threads the reference can use: its data path for one vhost controller
    # (= one LUN here) runs on exactly one reactor core (vhost_scsi.c:1311-1318), so a job of N LUNs - one per
    # GPU in our arm - keeps N cores busy.  --ref-procs overrides (e.g. to see what every core together does).
    nproc = cpu_reactor_count(args.ref_procs or max(1, args.gpus))
    farm = CpuFarm(nproc, 8, "randread")
    totals, singles = [], []
    for i in range(args.warmup + args.steps):
        vals, info = farm.run(per_step)
        if i >= args.warmup:
            totals.append(sum(vals))
            singles.append(statistics.mean(vals))
    farm.close()
    v = statistics.mean(totals)
    info = {**info, "cores": nproc,
            "sample": f"{nproc} reference reactors side by side (one process, one vhost controller + 8 GiB Malloc bdev each, as "
                      f"SPDK scales: one reactor per core), each: " + info["sample"],
            "per_core_value": statistics.mean(singles)}
    line = {"impl": "reference", "metric": "4KiB rand-read IOPS", "value": v, "unit": "IOPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"C2: 8 GiB Malloc bdev, 4 KiB random read, reference CPU poller x {nproc} reactors (cores)"},
            "cpu_baseline": {**info, "value": v},
            "e2e": {"value": v, "unit": "IOPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------

def device_pattern_fill(lun, store_ptr: int, nbytes: int, seed: int, torch):
    """prefill the backing store with the position-keyed pattern, generated on the GPU in 256 MiB
    chunks (same function as traces.pattern_words, in int64 two's-complement arithmetic)."""
    chunk_words = (256 << 20) // 8
    gamma = -7046029254386353131          # 0x9E3779B97F4A7C15 as int64
    m1, m2 = -4658895280553007687, -7723592293110705685

    def lsr(x, k):
        return (x >> k) & ((1 << (64 - k)) - 1)
    done = 0
    while done < nbytes // 8:
        n = min(chunk_words, nbytes // 8 - done)
        idx = torch.arange(done, done + n, dtype=torch.int64, device="cuda")
        z = (idx ^ seed) * gamma + gamma
        z = (z ^ lsr(z, 30)) * m1
        z = (z ^ lsr(z, 27)) * m2
        z = z ^ lsr(z, 31)
        torch.cuda.synchronize()
        lun.copy(store_ptr + done * 8, z.data_ptr(), n * 8)
        lun.sync()
        done += n


def pattern_fill_tensor(t, seed: int, torch):
    """fill a uint8 CUDA tensor (length a multiple of 8) with traces.pattern_words(seed, 0, ...) in place"""
    gamma = -7046029254386353131
    m1, m2 = -4658895280553007687, -7723592293110705685

    def lsr(x, k):
        return (x >> k) & ((1 << (64 - k)) - 1)
    words = t.view(torch.int64)
    chunk = (256 << 20) // 8
    for done in range(0, words.numel(), chunk):
        n = min(chunk, words.numel() - done)
        idx = torch.arange(done, done + n, dtype=torch.int64, device=t.device)
        z = (idx ^ seed) * gamma + gamma
        z = (z ^ lsr(z, 30)) * m1
        z = (z ^ lsr(z, 27)) * m2
        words[done:done + n] = z ^ lsr(z, 31)
        del idx, z


def nvlink_peak():
    """GB/s per direction per GPU that a peer copy reaches on this pool (B200_PROFILING.md: measured 770, nominal 900);
    profiles/nvlink.json (tools/nvlink_probe.cu on this pool) overrides when present"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "nvlink.json")))
        return float(d["ce_peer_copy_gbs"]), "measured (profiles/nvlink.json, tools/nvlink_probe.cu: copy-engine peer copy)"
    except (OSError, KeyError, ValueError):
        return 770.0, "B200_PROFILING.md: measured peer copy 770 GB/s per direction (900 nominal)"


def mirror_leg(args, rank, world, local, lib, torch, timer, barrier, max_over_ranks):
    """BASELINE config 5: 2-way mirrored bdev, 128 KiB sequential write, write fan-out over NVLink.
    One process per GPU: rank r is the PRIMARY of mirror r (store on its own GPU) and hosts the REPLICA of mirror r-1,
    which rank r-1 reaches through a CUDA IPC mapping; the mover warps store every unit twice, to local HBM and by P2P
    stores to the peer.  Two shapes: `pairs` - only even ranks write (N=2: one mirrored volume, N=4: two: SURVEY 8(d)
    C5 literally) - and `ring` - every rank writes, every NVLink port carries one replica stream out and one in.
    No reference implementation exists (S/lib/bdev/raid/bdev_raid.c:848-851 is RAID0 only), so parity is the contract
    of SURVEY 8(c): every replica equals what the single-bdev oracle holds after the same write trace - checked here
    on all 8 GiB of both replicas through position-keyed digests, and byte for byte against the oracle on a window."""
    import torch.distributed as dist
    nb = NUM_BLOCKS
    hosted = lib.construct_malloc_bdev(nb, BLOCK, name=f"MirrorReplica{rank}", device=local)
    ht = torch.frombuffer(bytearray(lib.bdev_export_store(hosted)), dtype=torch.uint8).cuda()
    handles = [torch.empty_like(ht) for _ in range(world)]
    dist.all_gather(handles, ht)
    right, left = (rank + 1) % world, (rank - 1) % world
    mname = lib.construct_mirror_bdev_remote(nb, BLOCK, local, [bytes(handles[right].cpu().numpy())], name=f"Mirror{rank}")
    ctrlr = f"mirror.{rank}"
    lib.construct_vhost_scsi_controller(ctrlr)
    lib.add_vhost_scsi_lun(ctrlr, 0, mname)
    sq, sp = args.seq_queues, args.seq_per_queue
    n = sq * sp
    t = traces.uniform_trace(n, nb, io_blocks=256, pattern="seqwrite", sg="pages", seed=0xC5000000 + rank)
    assert n * 131072 == nb * BLOCK, "one step = one full pass over the device"
    arena = torch.empty(t.arena_bytes, dtype=torch.uint8, device="cuda")
    pattern_fill_tensor(arena, 0xC5000000 + rank, torch)
    d_reqs = torch.from_numpy(t.reqs.view(np.uint8)).cuda()
    d_iovs = torch.from_numpy(t.bind(arena.data_ptr()).view(np.uint8)).cuda()
    d_cpls = torch.zeros(n * 48, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    res = {}
    with lib.Lun(ctrlr, 0, num_queues=sq, queue_size=32) as lun:
        def step():
            lun.submit_batch(sq, sp, d_reqs.data_ptr(), d_iovs.data_ptr(), len(t.iovs), d_cpls.data_ptr(), abi.MEM_DEVICE)
        for shape in ("pairs", "ring"):
            writer = shape == "ring" or rank % 2 == 0
            writers = world if shape == "ring" else (world + 1) // 2
            for _ in range(args.warmup):
                if writer:
                    step()
            lun.sync()
            barrier()
            timer.start(lun)
            for _ in range(args.steps):
                if writer:
                    step()
            timer.stop(lun)
            lun.sync()
            barrier()
            ms = max_over_ranks(timer.elapsed_ms() if writer else 0.0)
            gbs = writers * n * args.steps * 131072 / (ms / 1e3) / 1e9
            res[shape] = {"value": gbs, "unit": "GB/s of user writes, whole job", "mirrored_volumes": writers,
                          "per_volume_gbs": gbs / writers, "ms_per_step": ms / args.steps}
        c = np.frombuffer(d_cpls.cpu().numpy().tobytes(), dtype=abi.cpl_dtype)
        assert not c["status"].any() and (c["used_len"] == 108).all(), "mirror leg: bad completions"
        launches = lun.iostat()["kernel_launches"]
    # ---- parity, every byte of both replicas of every mirror ----
    barrier()
    mine = lib.digest_device(local, arena.data_ptr(), arena.numel())       # store == arena after a full sequential pass
    dg = torch.tensor([mine[0] & 0x7FFFFFFFFFFFFFFF, mine[1] & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device="cuda")
    all_dg = [torch.empty_like(dg) for _ in range(world)]
    dist.all_gather(all_dg, dg)
    prim = lib.bdev_digest(mname, 0)
    repl = lib.bdev_digest(hosted, 0)
    assert prim == mine, f"rank {rank}: primary store differs from the written payload"
    want_left = tuple(int(x) for x in all_dg[left].cpu())
    assert (repl[0] & 0x7FFFFFFFFFFFFFFF, repl[1] & 0x7FFFFFFFFFFFFFFF) == want_left, \
        f"rank {rank}: the replica of mirror {left} hosted here differs from what rank {left} wrote"
    oracle_window = None
    if rank == 0:
        # the oracle as CHECKER (never measured): the first 512 requests of the trace cover exactly the first 64 MiB
        from oracle import bindings
        try:
            bindings.build()
        except Exception:  # noqa: BLE001
            pass
        wreq, wblk = 512, 512 * 256
        o = bindings.PortOracle(wblk, BLOCK)
        harena = arena[:wreq * 131072].cpu().numpy()
        sub = traces.Trace(t.reqs[:wreq].copy(), t.iovs[:wreq * 32].copy(), harena.size)
        oc = o.submit(sub.reqs, sub.bind(harena.ctypes.data))
        assert not oc["status"].any()
        want = o.store.copy()
        o.close()
        for rep in (0, 1):
            got = lib.bdev_read_raw(mname, 0, wblk * BLOCK, replica=rep)
            assert (got == want).all(), f"replica {rep} differs from the oracle's store on the first 64 MiB"
        oracle_window = "first 64 MiB (512 requests) of both replicas of mirror 0 == oracle (C restatement) store, byte for byte"
    barrier()
    lib.remove_vhost_scsi_target(ctrlr, 0)
    lib.remove_vhost_controller(ctrlr)
    lib.delete_bdev(mname)
    barrier()                                   # every importer is gone before an exporter frees its store
    lib.delete_bdev(hosted)
    del arena, d_reqs, d_iovs, d_cpls
    torch.cuda.empty_cache()
    nv, nv_src = nvlink_peak()
    for shape in res:
        res[shape]["nvlink_frac"] = res[shape]["per_volume_gbs"] / nv    # R=2: one payload stream out of the primary
    return {"metric": "128KiB seq-write GB/s on 2-way mirrored bdevs (32 x 4 KiB SG pages), replica on the next GPU, fan-out "
                      "by P2P stores from the mover warps (oim_lun_queue_mirror_kernel)",
            **res, "replicas": 2, "nvlink_peak_gbs": nv, "nvlink_peak_source": nv_src, "gpu_launches": launches,
            "requests_per_step_per_volume": n,
            "parity": "digest(primary) == digest(replica on the peer GPU) == digest(written payload) over all 8 GiB of every "
                      "mirror (oimgpu_bdev_digest); " + (oracle_window or ""),
            "transport": "cross-process: replica store exported with cudaIpcGetMemHandle, imported by the primary's process"}


def run_ours(args, rank, world, local):
    # host side of the PCIe paths: this rank's CPU threads and pinned memory on the GPU's own NUMA node
    from oim_b200 import hostmem
    placement = hostmem.bind_to_gpu_node(local) if not args.no_numa else {"note": "--no-numa"}
    import torch
    torch.cuda.set_device(local)
    torch.zeros(1, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from oim_b200 import build, lib
    build.build()
    lib.init([local])
    peak, peak_src = peaks()

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    plan = shard_plan(rank, world)
    bname = lib.construct_malloc_bdev(NUM_BLOCKS, BLOCK, name=plan["bdev"], device=local)
    lib.construct_vhost_scsi_controller(plan["ctrlr"])
    lib.add_vhost_scsi_lun(plan["ctrlr"], plan["target"], bname)
    store_ptr = lib.get_bdevs(bname)[0]["device_ptr"]
    nq, per_q = args.queues, args.per_queue
    # two handles on the same target: the resident legs use caller-owned HBM arrays (tiny rings),
    # the e2e leg uses the library's host-visible rings
    lun = lib.Lun(plan["ctrlr"], plan["target"], num_queues=max(nq, args.seq_queues, 1024), queue_size=32)
    lun_e2e = lib.Lun(plan["ctrlr"], plan["target"], num_queues=args.e2e_queues, queue_size=1024)
    device_pattern_fill(lun, store_ptr, NUM_BLOCKS * BLOCK, plan["store_seed"], torch)
    timer = lib.Timer()
    out = {}

    def resident_leg(io_blocks, pattern, sg, nq, per_q, steps, warmup, check, target=0, dump=None):
        n = nq * per_q
        t = traces.uniform_trace(n, NUM_BLOCKS, io_blocks=io_blocks, pattern=pattern, sg=sg, seed=plan["trace_seed"],
                                 target=target)
        arena = torch.empty(t.arena_bytes, dtype=torch.uint8, device="cuda")
        if "write" in pattern:
            arena.view(torch.int64)[:] = 0x0123456789ABCDEF
        else:
            arena.zero_()
        d_reqs = torch.from_numpy(t.reqs.view(np.uint8)).cuda()
        d_iovs = torch.from_numpy(t.bind(arena.data_ptr()).view(np.uint8)).cuda()
        d_cpls = torch.zeros(n * 48, dtype=torch.uint8, device="cuda")
        k = len(t.iovs) // n

        def step():
            # one C call: queue q <- requests [q*per_q, (q+1)*per_q); everything already in HBM
            lun.submit_batch(nq, per_q, d_reqs.data_ptr(), d_iovs.data_ptr(), len(t.iovs), d_cpls.data_ptr(),
                             abi.MEM_DEVICE)
        for _ in range(warmup):
            step()
        lun.sync()
        barrier()
        l0 = lun.iostat()["kernel_launches"]
        timer.start(lun)
        for _ in range(steps):
            step()
        timer.stop(lun)
        lun.sync()
        barrier()
        ms = max_over_ranks(timer.elapsed_ms())
        launches = lun.iostat()["kernel_launches"] - l0
        c = np.frombuffer(d_cpls.cpu().numpy().tobytes(), dtype=abi.cpl_dtype)
        assert (c["status"] == 0).all() and (c["resid"] == 0).all() and (c["used_len"] > 0).all(), "bad completions"
        if check:
            check(t, arena)
        if dump and args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, dump, t, arena, c, torch)
        del arena, d_reqs, d_iovs, d_cpls
        torch.cuda.empty_cache()
        return n, ms, launches, t

    def check_randread(t, arena):
        # EVERY payload byte against the position-keyed pattern of the store: request i must hold the 512 words that
        # start at word lba_i * 64 (computed on the GPU, 2^17 requests at a time)
        cdb = torch.from_numpy(np.ascontiguousarray(t.reqs["cdb"][:, 2:6])).cuda().to(torch.int64)
        lba = (cdb[:, 0] << 24) | (cdb[:, 1] << 16) | (cdb[:, 2] << 8) | cdb[:, 3]
        gamma, m1, m2 = -7046029254386353131, -4658895280553007687, -7723592293110705685

        def lsr(x, k):
            return (x >> k) & ((1 << (64 - k)) - 1)
        words = arena.view(torch.int64).view(-1, 512)
        j = torch.arange(512, dtype=torch.int64, device="cuda")[None, :]
        for a in range(0, len(t.reqs), 1 << 17):
            idx = lba[a:a + (1 << 17), None] * 64 + j
            z = (idx ^ plan["store_seed"]) * gamma + gamma
            z = (z ^ lsr(z, 30)) * m1
            z = (z ^ lsr(z, 27)) * m2
            z = z ^ lsr(z, 31)
            bad = (words[a:a + (1 << 17)] != z).any(dim=1)
            assert not bool(bad.any()), f"request {a + int(bad.nonzero()[0])}: payload differs from the store pattern"
            del idx, z, bad

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n, ms, launches, _ = resident_leg(8, "randread", "single", nq, per_q, args.steps, args.warmup, check_randread,
                                      dump="rand4k")
    iops = aggregate(n, args.steps, world, ms)
    per_launch_ms = ms / max(1, launches)
    achieved = 2 * 4096 * n / (per_launch_ms / 1e3) / 1e9
    out["rand4k"] = (iops, ms / args.steps, launches)

    # ---- what a guest with 1 .. 254 request queues gets (and 1024 library rings, beyond what vhost-user can carry) ----
    sweep = None
    if not args.no_sweep:
        sweep = {"workload": "4 KiB random read, everything resident in HBM, 2^20 requests per step spread over Q request "
                             "queues, one launch per step; with fewer queues than the GPU holds CTAs (296) the CTAs share "
                             "the queues a pass of 32 at a time (KickHeader::shared)", "queues": {}}
        s0 = lun.shared_launches
        for q in (1, 2, 4, 8, 16, 64, 254, 1024):
            pq = max(32, (1 << 20) // q // 32 * 32)
            sn, sms, _, _ = resident_leg(8, "randread", "single", q, pq, max(3, args.steps // 2), 2, None)
            v = aggregate(sn, max(3, args.steps // 2), world, sms)
            sweep["queues"][str(q)] = {"value": v, "unit": "IOPS", "hbm_frac": 2 * 4096 * v / world / 1e9 / peak,
                                       "requests_per_step": sn}
        sweep["shared_queue_launches"] = lun.shared_launches - s0

    # ---- e2e: host request arrays through the C ABI, client buffers in pinned host memory ----
    e2e = None
    if not args.no_e2e:
        eq, ep = args.e2e_queues, args.e2e_per_queue
        en = eq * ep
        t = traces.uniform_trace(en, NUM_BLOCKS, io_blocks=8, pattern="randread", seed=plan["e2e_seed"])
        host = torch.empty(t.arena_bytes, dtype=torch.uint8).pin_memory()

        def pinned_like(a: np.ndarray) -> np.ndarray:
            """same contents in pinned host memory (a front end builds its requests there)"""
            buf = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
            out = buf.numpy().view(a.dtype)
            out[:] = a
            out_keep.append(buf)
            return out
        out_keep = []
        reqs_p = pinned_like(t.reqs)
        iovs = pinned_like(t.bind(host.data_ptr()))
        cpls = pinned_like(np.zeros(en, dtype=abi.cpl_dtype))
        L = lib.load()

        def e2e_step():
            # host->device: request + SG arrays (copy engine); device->host: payload (stored by the
            # movers into the pinned client buffers) + completion records (copy engine)
            rc = L.oimgpu_submit_and_wait(lun_e2e.h, eq, ep, reqs_p.ctypes.data, iovs.ctypes.data, len(iovs),
                                          cpls.ctypes.data, abi.MEM_HOST)
            assert rc == 0, rc
            return int(cpls["status"].sum()) + int((cpls["used_len"] != 4096 + 108).sum())
        for _ in range(max(1, args.warmup)):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            assert e2e_step() == 0
        barrier()
        wall = max_over_ranks(time.perf_counter() - t0)
        # device share of one step (explains the number; not part of it)
        timer.start(lun_e2e)
        L.oimgpu_submit_batch(lun_e2e.h, eq, ep, reqs_p.ctypes.data, iovs.ctypes.data, len(iovs), cpls.ctypes.data, abi.MEM_HOST)
        timer.stop(lun_e2e)
        lun_e2e.sync()
        dev_ms = timer.elapsed_ms()
        # every payload byte that arrived in the pinned client buffers, against the store's pattern
        elba = np.array([int.from_bytes(bytes(x[2:6]), "big") for x in t.reqs["cdb"]], dtype=np.uint64)
        ew = (elba[:, None] * np.uint64(64) + np.arange(512, dtype=np.uint64)[None, :]).reshape(-1)
        with np.errstate(over="ignore"):
            want = traces.mix64((np.uint64(plan["store_seed"]) ^ ew) * traces.GAMMA + traces.GAMMA)
        assert (host.numpy().view(np.uint64) == want).all(), "e2e payload differs from the store pattern"
        del ew, want
        # the box's host-side ceiling with every rank storing into host memory at once (explains e2e at N > 1)
        probe = hostmem.concurrent_d2h_probe(torch, local, barrier)
        if world > 1:
            import torch.distributed as dist
            tt = torch.tensor([probe["copy_engine_gbs"], probe["sm_stores_gbs"]], dtype=torch.float64, device="cuda")
            allp = [torch.empty_like(tt) for _ in range(world)]
            dist.all_gather(allp, tt)
            per_rank = [[float(x[0]), float(x[1])] for x in allp]
        else:
            per_rank = [[probe["copy_engine_gbs"], probe["sm_stores_gbs"]]]
        ceiling = {"copy_engine_gbs_total": sum(p[0] for p in per_rank), "sm_stores_gbs_total": sum(p[1] for p in per_rank),
                   "copy_engine_gbs_per_gpu": [round(p[0], 1) for p in per_rank], "sm_stores_gbs_per_gpu": [round(p[1], 1) for p in per_rank],
                   "how": "all ranks at once for 0.4 s each: cudaMemcpyAsync D2H and oim_copy_kernel stores of 256 MiB into this rank's "
                          "pinned buffer (oim_b200/hostmem.py; tools/pcie_concurrent_probe.py runs the same with and without binding)"}
        e2e = {"value": en * args.steps * world / wall, "unit": "IOPS", "host_placement": placement, "host_ceiling": ceiling,
               "h2d_bytes_per_step": int(en * 64 + len(iovs) * 16),
               "d2h_bytes_per_step": int(en * 4096 + en * 48),
               "ms_per_step": wall / args.steps * 1e3, "requests_per_step": en, "queues": eq,
               "device_ms_per_step": dev_ms, "pcie_payload_gbs_device": en * 4096 / (dev_ms / 1e3) / 1e9,
               "note": "host request/SG arrays in pinned memory -> copy-engine upload -> kernel on HBM-resident "
                       "metadata; payload stored by the movers straight into pinned client buffers over PCIe; "
                       "completion records copied back; host_ceiling = what the box's host side takes with every rank storing at "
                       "once (copy engine / SM stores), measured in this run"}

    # ---- virtqueue mode: the kernel walks real virtio split rings itself (a19-a22 on the device) ----
    vq = None
    if not args.no_vq:
        from oim_b200 import vring
        vnq, vper, vring_size = 4096, 256, 1024
        g = vring.build_uniform_queues(vnq, vper, NUM_BLOCKS, ring_size=vring_size, seed=plan["trace_seed"] + 5)
        guest = torch.empty(g.total_bytes(), dtype=torch.uint8, device="cuda")
        guest[:g.data_off] = torch.from_numpy(g.arena).cuda()
        guest[g.data_off:].zero_()
        gbase = guest.data_ptr()
        vlun = lib.Lun(plan["ctrlr"], plan["target"], num_queues=vnq, queue_size=32)
        vlun.set_mem_table(np.array([g.gpa_base, g.total_bytes(), gbase], dtype=np.uint64))
        for q in range(vnq):
            qb = gbase + q * g.q_stride
            vlun.vq_attach(q, qb + g.desc_off, qb + g.avail_off, qb + g.used_off, vring_size, 0, 0)
        # the guests' avail->idx fields, one u16 per queue, as a strided view
        avail_idx = guest[:g.data_off].view(torch.int16).view(vnq, g.q_stride // 2)[:, (g.avail_off + 2) // 2]
        used_idx = guest[:g.data_off].view(torch.int16).view(vnq, g.q_stride // 2)[:, (g.used_off + 2) // 2]

        def vstep():
            avail_idx.add_(vper)                     # every guest publishes vper more heads ...
            torch.cuda.current_stream().synchronize()
            vlun.vq_kick()                           # ... and kicks
        for _ in range(args.warmup):
            vstep()
        vlun.sync()
        barrier()
        vt = 0.0
        for _ in range(args.steps):
            avail_idx.add_(vper)
            torch.cuda.current_stream().synchronize()
            timer.start(vlun)
            vlun.vq_kick()
            timer.stop(vlun)
            vlun.sync()
            vt += timer.elapsed_ms()
        barrier()
        vms = max_over_ranks(vt)
        want_used = (vper * (args.steps + args.warmup)) & 0xFFFF
        assert int((used_idx.to(torch.int32) & 0xFFFF).min()) == want_used and int((used_idx.to(torch.int32) & 0xFFFF).max()) == want_used
        i = int(g.lba[3, 7])
        got = guest[g.data_off + (3 * vper + 7) * 4096:g.data_off + (3 * vper + 7) * 4096 + 4096].cpu().numpy()
        assert (got == traces.pattern_bytes(plan["store_seed"], i * BLOCK, 4096)).all(), "virtqueue payload mismatch"
        viops = aggregate(vnq * vper, args.steps, world, vms)
        vq = {"metric": "4KiB rand-read IOPS through guest virtio split rings (3-descriptor chains, ring walk, "
                        "GPA->VA translation, response + used ring written by the kernel)",
              "value": viops, "unit": "IOPS", "hbm_frac": 2 * 4096 * viops / world / 1e9 / peak,
              "queues": vnq, "requests_per_kick": vnq * vper}
        vlun.close()
        del guest
        torch.cuda.empty_cache()

        # ---- the resident poller as the measured path (north star K4): the same rings-in-HBM shape served by the
        # persistent kernel (doorbell = the guest's avail->idx, no launch per kick), next to one launch per kick on
        # the identical layout.  INDIRECT descriptors, 1024 requests per ring and round: a round is 2^22 requests.
        if not args.no_poller_leg:
            pq, pper = 4096, 1024
            g2 = vring.build_uniform_queues(pq, pper, NUM_BLOCKS, ring_size=1024, seed=plan["trace_seed"] + 6, indirect=True)
            guest = torch.empty(g2.total_bytes(), dtype=torch.uint8, device="cuda")
            meta_d = torch.from_numpy(g2.arena).cuda()
            res = {}
            for pmode in ("launch_per_kick", "resident_poller"):
                guest[:g2.data_off] = meta_d
                guest[g2.data_off:].zero_()
                gb = guest.data_ptr()
                plun = lib.Lun(plan["ctrlr"], plan["target"], num_queues=pq, queue_size=32)
                plun.set_mem_table(np.array([g2.gpa_base, g2.total_bytes(), gb], dtype=np.uint64))
                for q in range(pq):
                    qb = gb + q * g2.q_stride
                    plun.vq_attach(q, qb + g2.desc_off, qb + g2.avail_off, qb + g2.used_off, 1024, 0, 0)
                torch.cuda.synchronize()
                if pmode == "resident_poller":
                    plun.start_poller(idle_timeout_ms=20000)
                tot, rounds = 0.0, max(3, args.steps // 2)
                try:
                    for k in range(2 + rounds):
                        want = (pper * (k + 1)) & 0xFFFF

                        def used_all():
                            # the copy engine gathers the 4096 used indices: a torch kernel could not run next to the
                            # resident poller, which holds every SM slot
                            u = lib.read_strided(local, gb + g2.used_off + 2, g2.q_stride, 2, pq).view("<u2")
                            return bool((u == want).all())
                        # every guest publishes a ring full of heads: avail->idx += 1024, written by the copy engine too
                        lib.write_strided(local, gb + g2.avail_off + 2, np.full(pq, want, dtype="<u2"), g2.q_stride, 2)
                        t0 = time.perf_counter()
                        if pmode == "launch_per_kick":
                            plun.vq_kick()
                            plun.sync()
                        else:
                            while not used_all():
                                if time.perf_counter() - t0 > 30:
                                    raise TimeoutError("resident poller: completions missing")
                        dt = time.perf_counter() - t0
                        if k >= 2:
                            tot += dt
                        assert used_all()
                finally:
                    if pmode == "resident_poller":
                        plun.stop_poller()
                    plun.close()
                tot = max_over_ranks(tot)
                v = aggregate(pq * pper, rounds, world, tot * 1e3)
                res[pmode] = {"value": v, "unit": "IOPS", "hbm_frac": 2 * 4096 * v / world / 1e9 / peak, "ms_per_round": tot / rounds * 1e3}
            i = int(g2.lba[5, 9])
            got = guest[g2.data_off + (5 * pper + 9) * 4096:g2.data_off + (5 * pper + 9) * 4096 + 4096].cpu().numpy()
            assert (got == traces.pattern_bytes(plan["store_seed"], i * BLOCK, 4096)).all(), "poller leg payload mismatch"
            vq["resident_poller_hbm"] = {**res, "queues": pq, "requests_per_round": pq * pper,
                                         "timing": "host wall clock: avail->idx of every ring bumped on the device, then kick + sync "
                                                   "(launch per kick) or the host polling the used indices in HBM (resident poller: "
                                                   "each poll costs ~50 us, <1 % of a round)",
                                         "layout": "4096 virtqueues of 1024 INDIRECT descriptors in HBM, 2^22 requests per round"}
            del guest, meta_d
            torch.cuda.empty_cache()

    # ---- config 4 shape: mixed 70/30 random read/write, qd=128 per queue (bdevperf -M 70 -q 128) ----
    mixed = None
    if not args.no_mixed:
        mq, mp = 254, 4128                       # ~2^20 requests per step on the 254 queues a controller can carry; queue q stays inside LBA window q
        mt = traces.partitioned_queues(mq, mp, NUM_BLOCKS, pattern="randrw", read_pct=70, io_blocks=8, seed=plan["trace_seed"] + 99)
        marena = torch.empty(mt.arena_bytes, dtype=torch.uint8, device="cuda")
        marena.view(torch.int64)[:] = 0x5A5A5A5A5A5A5A5A
        m_reqs = torch.from_numpy(mt.reqs.view(np.uint8)).cuda()
        m_iovs = torch.from_numpy(mt.bind(marena.data_ptr()).view(np.uint8)).cuda()
        m_cpls = torch.zeros(len(mt.reqs) * 48, dtype=torch.uint8, device="cuda")
        for _ in range(args.warmup):
            lun.submit_batch(mq, mp, m_reqs.data_ptr(), m_iovs.data_ptr(), len(mt.iovs), m_cpls.data_ptr(), abi.MEM_DEVICE)
        lun.sync()
        barrier()
        timer.start(lun)
        for _ in range(args.steps):
            lun.submit_batch(mq, mp, m_reqs.data_ptr(), m_iovs.data_ptr(), len(mt.iovs), m_cpls.data_ptr(), abi.MEM_DEVICE)
        timer.stop(lun)
        lun.sync()
        barrier()
        mms = max_over_ranks(timer.elapsed_ms())
        mc = np.frombuffer(m_cpls.cpu().numpy().tobytes(), dtype=abi.cpl_dtype)
        assert not mc["status"].any()
        miops = aggregate(len(mt.reqs), args.steps, world, mms)
        mixed = {"metric": "4KiB 70/30 rand r/w IOPS (qd=128 per queue: 4 passes of 32 in flight per queue, 254 queues, "
                           "queue q confined to LBA window q)", "value": miops, "unit": "IOPS",
                 "hbm_frac": 2 * 4096 * miops / world / 1e9 / peak, "requests_per_step": len(mt.reqs),
                 "reads": mt.meta["reads"]}
        del marena, m_reqs, m_iovs, m_cpls
        torch.cuda.empty_cache()

    # ---- latency-bound corner: ONE request queue, qd=32, closed loop (submit 32 -> wait -> submit 32 ...) ----
    lat = None
    if not args.no_lat:
        rounds = 300
        lt = traces.uniform_trace(32 * rounds, NUM_BLOCKS, io_blocks=8, pattern="randread", seed=plan["e2e_seed"] + 7)
        lbuf = torch.empty(lt.arena_bytes, dtype=torch.uint8).pin_memory()
        liov = lt.bind(lbuf.data_ptr())
        lat = {}
        lcpl = np.zeros(32, dtype=abi.cpl_dtype)
        Lc = lib.load()
        for mode in ("launch_per_kick", "persistent_poller"):
            lq = lib.Lun(plan["ctrlr"], plan["target"], num_queues=1, queue_size=64)
            if mode == "persistent_poller":
                lq.start_poller(idle_timeout_ms=5000)
            try:
                for phase in ("warm", "timed"):
                    t0 = time.perf_counter()
                    for r in range(rounds if phase == "timed" else 20):
                        # one C call per round trip: 32 requests in, 32 completions out
                        rc = Lc.oimgpu_submit_and_wait(lq.h, 1, 32, lt.reqs[r * 32:].ctypes.data, liov.ctypes.data,
                                                       len(liov), lcpl.ctypes.data, abi.MEM_HOST)
                        assert rc == 0 and not lcpl["status"].any()
                    dt = time.perf_counter() - t0
            finally:
                if mode == "persistent_poller":
                    lq.stop_poller()
                lq.close()
            lat[mode] = {"iops": 32 * rounds / dt, "us_per_round_trip": dt / rounds * 1e6}
        lat["workload"] = "1 queue, qd=32, 4 KiB random read, closed loop of oimgpu_submit_and_wait calls, pinned client buffers"

    # ---- second metric: 128 KiB sequential write ----
    seq = None
    if not args.no_seq:
        # BASELINE config 3: the volume is what oim-csi-driver's ceph path maps - construct_rbd_bdev (HBM-backed
        # here) - attached as a SECOND target of the same controller, the way MapVolume adds volumes; the same
        # session reaches it through lun[1] = 1
        rbd = lib.construct_rbd_bdev("rbd", f"bench-image-{rank}", BLOCK, NUM_BLOCKS * BLOCK, name=f"Ceph{rank}", device=local)
        lib.add_vhost_scsi_lun(plan["ctrlr"], 1, rbd)
        sq, sp = args.seq_queues, args.seq_per_queue       # 256 x 256 x 128 KiB = one pass over the 8 GiB device
        n2, ms2, l2, _ = resident_leg(256, "seqwrite", "pages", sq, sp, args.steps, args.warmup, None, target=1)
        assert lun.iostat(1)["bytes_written"] >= n2 * 131072, "the writes were not booked on the RBD volume"
        seq_gbs = n2 * args.steps * world * 131072 / (ms2 / 1e3) / 1e9
        seq = {"metric": "128KiB seq-write GB/s (32 x 4 KiB SG pages)", "value": seq_gbs, "unit": "GB/s",
               "ms_per_step": ms2 / args.steps, "hbm_frac": 2 * seq_gbs / world / peak,
               "requests_per_step": n2, "queues": sq,
               "volume": "construct_rbd_bdev (Ceph RBD emulated in HBM), target 1 of the benchmark controller"}

    # ---- SURVEY 8(d) C3: the same 128 KiB sequential write with the other two SG shapes ----
    seq_sg = None
    if not args.no_seq and not args.no_extra:
        seq_sg = {}
        for sg_name, label in (("single", "1 x 131072 B"),
                               ("unaligned", "33 elements: 100 B + 31 x 4096 B + 3996 B, one client buffer split at those "
                                             "bytes (each element continues its predecessor: the parser joins the run "
                                             "into one segment; client buffers aligned like the store)"),
                               ("unaligned+3", "the same 33 elements with every client buffer 3 bytes off the store's "
                                               "16-byte alignment: one segment per request, every unit realigned "
                                               "(bulk copy into shared memory, funnel shifts on the way out)"),
                               ("scattered", "the same 33 element lengths, but no element continues its predecessor in "
                                             "client memory (reverse placement): 33 segments per request with "
                                             "byte-granular heads and tails, source 8 bytes off the destination")):
            n5, ms5, _, _ = resident_leg(256, "seqwrite", sg_name, args.seq_queues, args.seq_per_queue, args.steps, args.warmup, None, target=1)
            g5 = n5 * args.steps * world * 131072 / (ms5 / 1e3) / 1e9
            seq_sg[sg_name] = {"value": g5, "unit": "GB/s", "hbm_frac": 2 * g5 / world / peak, "sg": label}

    # ---- the other two corners of the same shapes: 4 KiB random WRITE, 128 KiB sequential READ ----
    extra = None
    if not args.no_extra:
        n3, ms3, _, _ = resident_leg(8, "randwrite", "single", nq, per_q // 4, args.steps, args.warmup, None)
        w_iops = aggregate(n3, args.steps, world, ms3)
        n4, ms4, _, _ = resident_leg(256, "seqread", "pages", args.seq_queues, args.seq_per_queue, args.steps, args.warmup, None)
        r_gbs = n4 * args.steps * world * 131072 / (ms4 / 1e3) / 1e9
        extra = {"rand4k_write": {"value": w_iops, "unit": "IOPS", "hbm_frac": 2 * 4096 * w_iops / world / 1e9 / peak,
                                  "requests_per_step": n3, "note": "random LBAs over the whole device from 1024 queues"},
                 "seq128k_read": {"value": r_gbs, "unit": "GB/s", "hbm_frac": 2 * r_gbs / world / peak, "requests_per_step": n4}}

    # ---- config 5: mirrored bdev across GPUs (needs a peer: N >= 2) ----
    mirror = None
    if world >= 2 and not args.no_mirror:
        mirror = mirror_leg(args, rank, world, local, lib, torch, timer, barrier, max_over_ranks)

    clocks = sampler.stop() if rank == 0 else {}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # this configuration is ONE LUN behind one controller: the reference serves it from one reactor core
        leg = CpuLeg(8, "randread")
        v, info = leg.run(args.cpu_seconds)
        leg.close()
        cpu = {**info, "value": v}
        # the same reference as a vhost-user slave, driven by the master script of the `vhost_user` leg: the
        # like-for-like baseline of the path a VM takes (its transport, its poller, its memcpy; one reactor core)
        if not args.no_vu and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "liboim_ref_vhost.so")):
            try:
                cpu["vhost_user"] = vhost_user_leg(args, local, "reference")
            except Exception as e:  # noqa: BLE001
                cpu["vhost_user"] = {"error": f"{type(e).__name__}: {e}"[:300]}

    lun.close()
    lun_e2e.close()
    # ---- the path a VM takes: a separate daemon process, a vhost-user master, guest RAM in a shared memfd ----
    vuser = None
    if rank == 0 and world == 1 and not args.no_vu:
        try:
            counts = (1, 2, 4, 8, 16, 64, 254)
            vuser = {"launch_per_kick": vhost_user_leg(args, local, "kick", counts), "resident_poller": vhost_user_leg(args, local, "poller", counts),
                     "workload": "oim-gpu-vhost + vhost-user master over its socket: Q request queues (headline: 64; by_queues: 1..254, the "
                                 "most a vhost-scsi controller can carry) x 256 READ(10) of 4 KiB per round, 3-descriptor chains in guest "
                                 "RAM (host memory, pinned by the daemon), 1 GiB Malloc bdev"}
        except Exception as e:                          # a leg that cannot run must not cost the headline line
            vuser = {"error": f"{type(e).__name__}: {e}"[:300]}
    # ---- OIM's real attach shape on a multi-GPU box: ONE daemon owning all N GPUs, ONE controller with N targets (one
    # volume per GPU), ONE vhost-user session whose request queues are dealt out over the GPUs ----
    vuser_multi = None
    if world >= 2 and not args.no_vu:
        import torch.distributed as dist
        lib.fini()                                  # every rank lets go of its GPU's memory; rank 0's daemon takes all N GPUs
        torch.cuda.empty_cache()
        barrier()
        # the other ranks wait on the rendezvous store, on the CPU: an NCCL barrier would spin a kernel on their GPUs,
        # which are the daemon's GPUs for this leg
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                # INDIRECT descriptors (what a Linux guest uses): a 1024-entry ring then holds 1024 requests, so a round is
                # 260 096 requests = 1 GiB of payload and the control path (Python master, eventfds) weighs less
                one = vhost_user_leg(args, local, "kick", (254,), per_q=1024, indirect=True)
                allg = vhost_user_leg(args, local, "kick", (254,), gpus=list(range(world)), per_q=1024, indirect=True)
                vuser_multi = {"one_gpu_one_lun": one, f"{world}_gpus_{world}_luns_one_controller": allg,
                               "speedup": allg["value"] / one["value"],
                               "workload": f"one oim-gpu-vhost --gpus 0..{world - 1}, one controller, {world} targets (1 GiB Malloc bdev each, placed "
                                           "one per GPU), one vhost-user session with 254 request queues x 256 READ(10) of 4 KiB per round, requests "
                                           "dealt out over the targets; queue r is served by GPU r mod N (any GPU reaches any target: own HBM or "
                                           "a peer's over NVLink), so payload crosses all N PCIe links; single-process Python master; the guest's RAM is one "
                                           "registered memfd on one NUMA node: its host-side write ceiling (~86 GB/s on this pool's boxes, "
                                           "reached with 2 GPUs) bounds this leg, see DESIGN.md 6c'"}
            except Exception as e:  # noqa: BLE001
                vuser_multi = {"error": f"{type(e).__name__}: {e}"[:300]}
            store.set("oim_multi_gpu_leg_done", "1")
        else:
            store.wait(["oim_multi_gpu_leg_done"])
        barrier()
    if rank == 0:
        line = {
            "metric": "4KiB rand-read IOPS", "value": iops, "unit": "IOPS", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"C2: one 8 GiB HBM Malloc bdev per GPU, 4 KiB random read, qd=32 per request "
                                   f"queue x {nq} queues, {per_q} requests/queue/step",
                       "queues": nq, "per_queue": per_q, "requests_per_step_per_gpu": n,
                       "queue_limit": "254 request queues = the most one vhost-scsi controller can carry "
                                      "(S/lib/vhost/vhost_internal.h:63); queue_sweep has 1..1024",
                       "l2": "inputs larger than L2: 8 GiB store + unique 4 KiB client buffer per request "
                             f"({n * 4096 >> 20} MiB) per step"},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": measured_traffic("rand4k", n), "peak_source": peak_src,
                         "traffic_source": "ncu --set full capture, profiles/r2_rand4k_ncu.md (bytes per launch)",
                         "algorithmic_bytes_per_launch": 2 * 4096 * n, "kernel": "oim_lun_queue_kernel"},
            "seq128k": seq, "virtqueue": vq, "mixed_70_30": mixed, "e2e": e2e, "single_queue_qd32": lat, "cpu_baseline": cpu,
            "vhost_user": vuser, "more": extra, "mirror": mirror, "queue_sweep": sweep, "seq128k_sg": seq_sg, "vhost_user_multi_gpu": vuser_multi,
        }
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def vhost_user_leg(args, device: int, mode: str, queue_counts=(64,), gpus=None, daemon_args=(), env=None,
                   per_q: int = 256, indirect: bool = False) -> dict:
    """The path a VM takes: oim-gpu-vhost as a separate process, a vhost-user master (what QEMU is) connected
    to <socket dir>/scsi0, guest RAM in a shared memfd that the daemon pins for the GPU, 4 KiB random READs
    published on virtio rings and kicked through eventfds; completion = used index + call eventfd.
    Wall-clock around kick -> all completions seen (two processes: there is no common CUDA stream to time on).
    One daemon, one vhost-user session per entry of queue_counts (a guest with that many request queues);
    returns the 64-queue entry (or the only one) with the others under "by_queues"."""
    import json as _json
    import socket
    import subprocess
    import tempfile
    import time
    from oim_b200 import build, vhost_user_master as vu, vring

    ring = 1024
    max_q = max(queue_counts)
    nb = 1 << 21                                         # 1 GiB bdev: far larger than L2
    tmp = tempfile.mkdtemp(prefix="oimvu", dir="/tmp")        # socket paths must fit sun_path (108 bytes)
    os.mkdir(os.path.join(tmp, "vhost"))
    rpc = os.path.join(tmp, "rpc.sock")
    log = open(os.path.join(tmp, "daemon.log"), "wb")
    if mode == "reference":
        # the reference's own vhost target (S/lib/vhost incl. its vhost-user transport, compiled into oracle/_ref) as the
        # slave: one reactor core polling the rings, exactly what QEMU would talk to in an SPDK deployment
        cmd = [sys.executable, os.path.join(ROOT, "tests", "ref_rpc_server.py"), rpc, os.path.join(tmp, "vhost"), "vhost", "busy"]
    else:
        cmd = ([build.DAEMON, "-r", rpc, "-S", os.path.join(tmp, "vhost"), "--gpus", ",".join(str(x) for x in (gpus or [device]))] +
               (["--poller"] if mode == "poller" else []) + list(daemon_args))
    proc = subprocess.Popen(cmd, stdout=log, stderr=log, env={**os.environ, **(env or {})})
    try:
        t0 = time.time()
        while not os.path.exists(rpc):
            if proc.poll() is not None or time.time() - t0 > 120:
                raise RuntimeError("oim-gpu-vhost did not start: " + open(os.path.join(tmp, "daemon.log")).read()[-500:])
            time.sleep(0.02)
        c = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        for _ in range(500):             # (the reference's server binds first and listens a moment later)
            try:
                c.connect(rpc)
                break
            except (ConnectionRefusedError, FileNotFoundError):
                time.sleep(0.01)

        def call(i, method, params):
            c.sendall((_json.dumps({"jsonrpc": "2.0", "method": method, "params": params, "id": i}) + "\n").encode())
            buf = b""
            while not buf.endswith(b"\n"):
                buf += c.recv(65536)
            return _json.loads(buf)
        # OIM's shape (MapVolume, controller.go:131-148): ONE controller, every volume another target of it; with several
        # GPUs the daemon places the bdevs round-robin (least-loaded GPU) and deals the session's queues out over the GPUs
        ntgt = len(gpus) if gpus else 1
        assert call(2, "construct_vhost_scsi_controller", {"ctrlr": "scsi0"})["result"] is True
        for t in range(ntgt):
            assert call(10 + t, "construct_malloc_bdev", {"num_blocks": nb, "block_size": BLOCK, "name": f"M{t}"})["result"] == f"M{t}"
            assert call(30 + t, "add_vhost_scsi_lun", {"ctrlr": "scsi0", "scsi_target_num": t, "bdev_name": f"M{t}"})["result"] == t

        g = vring.build_uniform_queues(max_q, per_q, nb, ring_size=ring, seed=77, ntargets=ntgt, indirect=indirect)
        tail = 2 << 20                                   # control / event rings live behind the payload area
        total = -(-(g.total_bytes() + tail) // (2 << 20)) * (2 << 20)
        ram = vu.GuestRam(total)
        pristine = g.arena.copy()
        results = {}
        for nq in queue_counts:
            ram.mem[:g.data_off] = pristine              # fresh rings (avail/used indices back to 0) for a fresh session
            ram.mem[g.data_off:g.data_off + g.data_bytes] = 0xAA
            m = vu.Master(os.path.join(tmp, "vhost", "scsi0"), timeout=60)
            f = m.get_u64(vu.GET_FEATURES)
            m.set_u64(vu.SET_PROTOCOL_FEATURES, m.get_u64(vu.GET_PROTOCOL_FEATURES) & 0x9)
            m.send(vu.SET_OWNER)
            m.set_u64(vu.SET_FEATURES, f & ~(1 << vu.F_LOG_ALL))
            # one region: guest-physical gpa_base.. <-> memfd offset 0..; master VA = UVA_BASE + offset
            assert m.set_mem_table([(g.gpa_base, total, vu.UVA_BASE, 0, ram.fd)], need_reply=True) == 0
            t_off = g.total_bytes()
            queues = [vu.Queue(0, 16, t_off, t_off + 256, t_off + 320), vu.Queue(1, 16, t_off + 8192, t_off + 8192 + 256, t_off + 8192 + 320)]
            for q in range(nq):
                b = q * g.q_stride
                queues.append(vu.Queue(2 + q, ring, b + g.desc_off, b + g.avail_off, b + g.used_off))
            for q in queues:
                q.setup(m)
            time.sleep(0.5)
            a_off = [q * g.q_stride + g.avail_off + 2 for q in range(nq)]
            u_off = [q * g.q_stride + g.used_off + 2 for q in range(nq)]
            avail = [ram.mem[o:o + 2].view("<u2") for o in a_off]
            used = [ram.mem[o:o + 2].view("<u2") for o in u_off]

            def round_trip(k):
                want = (per_q * (k + 1)) & 0xFFFF
                for a in avail:
                    a[0] = want
                for q in queues[2:]:
                    q.notify()
                spin = time.perf_counter()
                while True:
                    if all(int(u[0]) == want for u in used):
                        return
                    if time.perf_counter() - spin > 60:
                        raise TimeoutError("vhost-user leg: completions missing")
            for k in range(args.warmup):
                round_trip(k)
            t0 = time.perf_counter()
            for k in range(args.steps):
                round_trip(args.warmup + k)
            dt = time.perf_counter() - t0
            payload = ram.mem[g.data_off:g.data_off + nq * per_q * 4096]
            assert not payload.any(), "a fresh Malloc bdev reads as zeros; the buffers were 0xAA"
            if nq < max_q:
                assert (ram.mem[g.data_off + nq * per_q * 4096:g.data_off + nq * per_q * 4096 + 4096] == 0xAA).all()
            el = ram.mem[g.used_off + 4:g.used_off + 4 + 8 * ring].view(vring.used_elem_dtype)
            assert int(el["len"][0]) == 108 + 4096
            for q in queues:
                m.get_vring_base(q.index)
            m.close()
            iops = nq * per_q * args.steps / dt
            for q in queues:
                q.close()
            del avail, used, payload, el
            results[nq] = {"value": iops, "unit": "IOPS", "mode": mode, "queues": nq, "requests_per_kick_round": nq * per_q,
                           "payload_gbs": iops * 4096 / 1e9, "ms_per_round": dt / args.steps * 1e3,
                           "timing": "host wall clock in the master process, kick -> every used index seen"}
            time.sleep(0.3)                              # the daemon notices the closed session before the next one connects
        ram.close()
        main_q = 64 if 64 in results else queue_counts[-1]
        out = dict(results[main_q])
        if len(results) > 1:
            out["by_queues"] = {str(k): {"value": v["value"], "payload_gbs": v["payload_gbs"], "ms_per_round": v["ms_per_round"]}
                                for k, v in results.items()}
        return out
    finally:
        proc.terminate()
        try:
            proc.wait(10)
        except Exception:
            proc.kill()
        log.close()


def main():
    args = parse_args()
    rank, world, local = dist_setup(args)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local)


if __name__ == "__main__":
    main()
