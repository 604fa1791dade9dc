"""The vhost-user transport (SURVEY.md 8(f) rank 2): a master - what QEMU's vhost-user-scsi-pci is - connects to
<socket dir>/<controller>, shares its memory, hands over the virtqueues and does I/O.

The same master script (oim_b200/vhost_user_master.py) runs against oim-gpu-vhost and against the REFERENCE'S OWN
transport + vhost-scsi + bdev stack (oracle/_ref/liboim_ref_vhost.so: S/lib/vhost/rte_vhost/* compiled where it
lies), and the protocol transcripts and the guest memory are compared.  The reference's side is stored
(tests/golden/reference/vhost_user.json.xz: transcripts, completions, digests of the guest memory; see tests/util.py).

CPU: handshake, control queue, event queue / hot-plug (our daemon with --control-only: no data path exists then).
GPU: request queues served by the kernel, launch-per-kick and resident-poller mode."""
import os
import struct
import subprocess
import sys
import time

import numpy as np
import pytest

import util
from oim_b200 import abi, traces, vring
from test_rpc_daemon import DAEMON, ROOT, Client
from oim_b200 import vhost_user_master as vu

META_END = 2 * vring.R01_SIZE + (4 << 20)          # end of the image's metadata area (rings, headers)
NB = 32768


class Slave:
    """one server process (ours or the reference) + its RPC client"""

    def __init__(self, kind: str, tmp, extra=()):
        self.kind = kind
        self.dir = tmp / kind
        (self.dir / "vhost").mkdir(parents=True)
        self.rpc = str(self.dir / "rpc.sock")
        self.log = open(self.dir / "log.txt", "wb")
        if kind == "ref":
            cmd = [sys.executable, os.path.join(ROOT, "tests", "ref_rpc_server.py"), self.rpc, str(self.dir / "vhost"), "vhost"]
        else:
            cmd = [DAEMON, "-r", self.rpc, "-S", str(self.dir / "vhost"), *extra]
        self.p = subprocess.Popen(cmd, stdout=self.log, stderr=self.log)
        t0 = time.time()
        while not os.path.exists(self.rpc):
            assert self.p.poll() is None, f"{kind} server died: {open(self.dir / 'log.txt').read()[-2000:]}"
            assert time.time() - t0 < 60
            time.sleep(0.01)
        self.c = Client(self.rpc)

    def call(self, method, params=None):
        return self.c.call(method, params)

    def sock(self, ctrlr):
        return str(self.dir / "vhost" / ctrlr)

    def close(self):
        if self.kind != "ref" and self.p.poll() is None:
            import signal
            self.p.send_signal(signal.SIGUSR2)             # every transport thread reports where it is
            time.sleep(0.3)
        self.p.terminate()
        try:
            self.p.wait(5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.log.close()


def provision(s: Slave):
    assert b'"result"' in s.call("construct_malloc_bdev", {"num_blocks": NB, "block_size": 512, "name": "M0"})
    assert b'"result"' in s.call("construct_malloc_bdev", {"num_blocks": 4096, "block_size": 512, "name": "M1"})
    assert b'"result":true' in s.call("construct_vhost_scsi_controller", {"ctrlr": "scsi0"})
    assert b'"result":0' in s.call("add_vhost_scsi_lun", {"ctrlr": "scsi0", "scsi_target_num": 0, "bdev_name": "M0"})


def small_ring(k: int):
    """(desc, avail, used, buffers) offsets of a 16-entry ring in the tail of the metadata area"""
    base = META_END - (k + 1) * 8192
    return base, base + 256, base + 320, base + 1024


def gpa_of(img, off):
    for g, s, o in img.regions:
        if o <= off < o + s:
            return off - o + g
    raise KeyError(off)


def put_chain(ram, img, ring, slot0, bufs):
    """descriptor chain in ring slots slot0.. : bufs = [(arena offset, len, writable)]; -> head"""
    d_off = ring[0]
    d = ram.mem[d_off:d_off + 16 * 16].view(vring.desc_dtype)
    for k, (off, ln, wr) in enumerate(bufs):
        last = k + 1 == len(bufs)
        d[slot0 + k] = (gpa_of(img, off), ln, (vring.F_WRITE if wr else 0) | (0 if last else vring.F_NEXT), 0 if last else slot0 + k + 1)
    return slot0


def publish(ram, ring, heads):
    a_off = ring[1]
    idx = int(ram.mem[a_off + 2:a_off + 4].view("<u2")[0])
    for h in heads:
        ram.mem[a_off + 4 + 2 * (idx % 16):a_off + 6 + 2 * (idx % 16)] = np.frombuffer(struct.pack("<H", h), np.uint8)
        idx += 1
    ram.mem[a_off + 2:a_off + 4] = np.frombuffer(struct.pack("<H", idx & 0xFFFF), np.uint8)


def handshake(m: vu.Master, ram, img, queues):
    f = m.get_u64(vu.GET_FEATURES)
    pf = m.get_u64(vu.GET_PROTOCOL_FEATURES)
    m.set_u64(vu.SET_PROTOCOL_FEATURES, pf & ((1 << vu.PF_MQ) | (1 << vu.PF_REPLY_ACK)))
    m.get_u64(vu.GET_QUEUE_NUM)
    m.get_config()
    m.send(vu.SET_OWNER)
    m.set_u64(vu.SET_FEATURES, f & ~(1 << vu.F_LOG_ALL), need_reply=True)
    regs = [(g, s, vu.UVA_BASE + o, o, ram.fd) for g, s, o in img.regions]
    assert m.set_mem_table(regs, need_reply=True) == 0
    for q in queues:                                    # in index order, as QEMU does
        q.setup(m)
        m.vring_state(vu.SET_VRING_ENABLE, q.index, 1)
    return f, pf


def control_requests(ram, img, ring):
    """task-management / async-notification requests on the control queue -> heads"""
    buf = ring[3]

    def req(slot, typ, sub, lun):
        o = buf + 64 * slot
        ram.mem[o:o + 24] = np.frombuffer(struct.pack("<II8sQ", typ, sub, bytes(lun), 0x1000 + slot), np.uint8)
        ram.mem[o + 32:o + 48] = 0xEE
        return o

    lun0, lun5, bad = [1, 0, 0, 0, 0, 0, 0, 0], [1, 5, 0, 0, 0, 0, 0, 0], [0, 0, 0, 0, 0, 0, 0, 0]
    heads = []
    o = req(0, 0, 5, lun0); heads.append(put_chain(ram, img, ring, 0, [(o, 24, 0), (o + 32, 1, 1)]))     # LUN RESET, present
    o = req(1, 0, 0, lun0); heads.append(put_chain(ram, img, ring, 2, [(o, 24, 0), (o + 32, 1, 1)]))     # ABORT TASK: unsupported
    o = req(2, 0, 5, lun5); heads.append(put_chain(ram, img, ring, 4, [(o, 24, 0), (o + 32, 1, 1)]))     # absent target
    o = req(3, 0, 5, bad); heads.append(put_chain(ram, img, ring, 6, [(o, 24, 0), (o + 32, 1, 1)]))      # malformed address
    o = req(4, 1, 0, lun0); heads.append(put_chain(ram, img, ring, 8, [(o, 24, 0), (o + 32, 5, 1)]))     # AN_QUERY
    o = req(5, 2, 0, lun0); heads.append(put_chain(ram, img, ring, 10, [(o, 24, 0), (o + 32, 4, 1)]))    # AN_SUBSCRIBE, short buffer
    o = req(6, 9, 0, lun0); heads.append(put_chain(ram, img, ring, 12, [(o, 24, 0), (o + 32, 1, 1)]))    # unknown type
    o = req(7, 0, 5, lun0); heads.append(put_chain(ram, img, ring, 14, [(o, 24, 0)]))                     # no response descriptor
    return heads


def event_buffers(ram, img, ring, n=4):
    heads = []
    for k in range(n):
        o = ring[3] + 32 * k
        ram.mem[o:o + 16] = 0xEE
        heads.append(put_chain(ram, img, ring, k, [(o, 16, 1)]))
    return heads


def wait_used(ram, ring, want, timeout=10.0):
    t0 = time.time()
    while time.time() - t0 < timeout:
        if int(ram.mem[ring[2] + 2:ring[2] + 4].view("<u2")[0]) == want:
            return
        time.sleep(0.002)
    raise TimeoutError(f"used idx {int(ram.mem[ring[2] + 2:ring[2] + 4].view('<u2')[0])}, wanted {want}")


def deliberate(log):
    """The one deliberate difference on the wire: dirty-page logging is not offered (VHOST_F_LOG_ALL, bit 26, and the
    LOG_SHMFD protocol feature, bit 1) - see vhost_user.cpp kFeatures.  Everything else must match the reference."""
    out = []
    for k, v in log:
        if k == vu.GET_FEATURES and v is not None:
            v &= ~(1 << 26)
        if k == vu.GET_PROTOCOL_FEATURES and v is not None:
            v &= ~(1 << 1)
        out.append((k, v))
    return out


def run_script(s: Slave, rq, *, data: bool, seed=5):
    """the whole life of one VM against one slave; -> (transcript, {label: guest memory snapshot})"""
    img = vring.build_image(rq if data else [], ring_size=256, seed=seed, mutate=False)
    ram = vu.GuestRam(img.arena.size)
    ram.mem[:] = img.arena
    cq, eq, q3 = small_ring(0), small_ring(1), small_ring(2)
    for r in (cq, eq, q3):
        ram.mem[r[0]:r[0] + 8192] = 0
    queues = [vu.Queue(0, 16, *cq[:3]), vu.Queue(1, 16, *eq[:3]), vu.Queue(2, img.ring_size, img.desc_off, img.avail_off, img.used_off),
              vu.Queue(3, 16, *q3[:3])]
    snaps = {}
    m = vu.Master(s.sock("scsi0"))
    try:
        handshake(m, ram, img, queues)
        # both slaves start the session asynchronously (ours pins the guest memory first)
        deadline, pending = time.time() + 10, list(queues)
        while pending and time.time() < deadline:
            pending = [q for q in pending if q.drain_calls() < 1]
            time.sleep(0.02)
        assert not pending, "every queue gets a spurious interrupt at start (vhost.c:1101-1115)"
        time.sleep(0.2)
        # ---- control queue
        publish(ram, cq, control_requests(ram, img, cq))
        queues[0].notify()
        wait_used(ram, cq, 8)
        # ---- event queue: hot-plug a second target, then remove it
        publish(ram, eq, event_buffers(ram, img, eq))
        queues[1].notify()
        assert b'"result":1' in s.call("add_vhost_scsi_lun", {"ctrlr": "scsi0", "scsi_target_num": 1, "bdev_name": "M1"})
        wait_used(ram, eq, 1)
        if data:
            # ---- request queues: the image's requests on queue 2, one READ of the hot-plugged target on queue 3
            o = q3[3]
            hdr = np.zeros(51, np.uint8)
            hdr[0:2] = [1, 1]
            hdr[19:51] = abi.cdb_rw(abi.READ_10, 8, 8)
            ram.mem[o:o + 51] = hdr
            ram.mem[o + 64:o + 64 + 108] = 0xEE
            data_off = META_END - 4 * 8192                # a spare page in the metadata area
            ram.mem[data_off:data_off + 4096] = 0x11
            publish(ram, q3, [put_chain(ram, img, q3, 0, [(o, 51, 0), (o + 64, 108, 1), (data_off, 4096, 1)])])
            queues[2].notify()
            queues[3].notify()
            queues[2].wait_used(ram, img.meta["placed"])
            queues[3].wait_used(ram, 1)
        assert b'"result":true' in s.call("remove_vhost_scsi_target", {"ctrlr": "scsi0", "scsi_target_num": 1})
        wait_used(ram, eq, 2)
        snaps["end"] = ram.mem.copy()
        for q in queues:
            m.get_vring_base(q.index)
        return m.log, snaps, img, (cq, eq, q3)
    finally:
        m.close()
        for q in queues:
            q.close()
        ram.close()


def mask(mem, img, rings):
    """what may differ between two correct slaves: the order of used-ring elements on the request queue
    (completion order is timing in the reference) and used->flags (the reference polls and sets NO_NOTIFY;
    a launch per kick needs the kick)"""
    c = img.masked(mem)
    for used_off in [img.used_off] + [r[2] for r in rings]:
        c[used_off:used_off + 2] = 0
    cq = rings[0]
    c[cq[2] + 4:cq[2] + 4 + 8 * 16] = 0       # control queue: the reference completes a LUN RESET asynchronously, i.e. last
    return c


def used_set(mem, ring, n):
    u = mem[ring[2] + 4:ring[2] + 4 + 8 * n].view(vring.used_elem_dtype)
    return sorted((int(i), int(l)) for i, l in u)


@pytest.fixture()
def slaves(oracles, sock_dir):
    from oim_b200 import build
    build.build()
    made = []

    def make(kind, extra=()):
        assert kind == "ours" or util.RECORD, "the reference slave runs only to record its side (util.reference_json)"
        s = Slave(kind, sock_dir, extra)
        made.append(s)
        provision(s)
        return s
    yield make
    for s in made:
        s.close()
        print(f"---- {s.dir.name} server log (tail) ----")           # shown by pytest when the test failed
        print(open(s.dir / "log.txt", errors="replace").read()[-3000:])


def reference_side(slaves, key: str, run):
    """what `run(reference slave)` returned, as stored (util.reference_json); in record mode from a live reference
    slave (the reference's own transport + vhost-scsi + bdev stack, oracle/_ref/liboim_ref_vhost.so)"""
    return util.reference_json("vhost_user", key, lambda: run(slaves("ref")))


def transcript(log):
    """a master's transcript back from its stored form (JSON lists)"""
    return tuple(log) if log and log[0] == "dropped" else [tuple(e) for e in log]


def assert_same_memory(got: np.ndarray, want, what="guest memory"):
    util.assert_same_digests(got, np.array(want, dtype=np.uint64), what)


def skip_without_gpu_after_recording():
    import torch
    if util.RECORD and not torch.cuda.is_available():
        pytest.skip("the reference's side is recorded; our side needs a GPU")


def test_vhost_user_handshake_control_and_event_queues(slaves):
    ours = slaves("ours", ["--control-only"])
    lo, so, img, rings = run_script(ours, [], data=False)

    def ref_run(ref):
        lr, sr, _, _ = run_script(ref, [], data=False)
        return {"log": lr, "mem": util.block_digests(mask(sr["end"], img, rings)).tolist(), "used_cq": used_set(sr["end"], rings[0], 8)}
    r = reference_side(slaves, "handshake", ref_run)
    lr = transcript(r["log"])
    assert deliberate(lo) == deliberate(lr), f"protocol transcripts differ:\nours {lo}\nref  {lr}"
    assert_same_memory(mask(so["end"], img, rings), r["mem"])
    # and the values themselves, so that two equally wrong slaves cannot pass
    d = dict((k, v) for k, v in lo if v is not None)
    assert d[vu.GET_FEATURES] == 0x150000007 and d[vu.GET_PROTOCOL_FEATURES] == 0x21D and d[vu.GET_QUEUE_NUM] == 128
    dr = dict((k, v) for k, v in lr if v is not None)
    assert dr[vu.GET_FEATURES] == 0x154000007 and dr[vu.GET_PROTOCOL_FEATURES] == 0x21F       # the reference's, for the record
    cq, eq, _ = rings
    resp = [int(so["end"][cq[3] + 64 * k + 32]) for k in range(8)]
    assert resp[:4] == [0, 2, 3, 3] and int(so["end"][cq[3] + 64 * 4 + 36]) == 2 and resp[6] == 0xEE
    assert used_set(so["end"], cq, 8) == [tuple(u) for u in r["used_cq"]] == [(0, 0), (2, 1), (4, 1), (6, 1), (8, 1), (10, 0), (12, 1), (14, 0)]
    ev = so["end"][eq[3]:eq[3] + 16].tobytes()
    assert struct.unpack("<I8sI", ev) == (1, bytes([1, 1, 0, 0, 0, 0, 0, 0]), 1)      # TRANSPORT_RESET, target 1, RESCAN
    ev2 = so["end"][eq[3] + 32:eq[3] + 48].tobytes()
    assert struct.unpack("<I8sI", ev2) == (1, bytes([1, 1, 0, 0, 0, 0, 0, 0]), 2)     # ... REMOVED


def test_remove_controller_with_a_master_connected_is_busy(slaves):
    """spdk_vhost_dev_unregister: "Controller %s has still valid connection" -> -EBUSY (S/lib/vhost/vhost.c:783-788); round 1
    tore the session down instead (ADVICE r1).  Same RPC replies from both servers, before and after the master leaves."""
    def run(s):
        for t in range(8):
            s.call("remove_vhost_scsi_target", {"ctrlr": "scsi0", "scsi_target_num": t})     # whatever provision() attached
        m = vu.Master(s.sock("scsi0"))
        m.get_u64(vu.GET_FEATURES)                       # the connection is established and served
        busy = s.call("remove_vhost_controller", {"ctrlr": "scsi0"})
        m.close()
        deadline = time.time() + 10
        while True:                                      # the slave notices the closed socket on its own thread
            r = s.call("remove_vhost_controller", {"ctrlr": "scsi0"})
            if b'"result":true' in r or time.time() > deadline:
                break
            time.sleep(0.05)
        return {"busy": busy.decode(), "last": r.decode(), "socket_left": os.path.exists(s.sock("scsi0"))}
    got = run(slaves("ours", ["--control-only"]))
    for kind, out in (("ours", got), ("ref", reference_side(slaves, "remove_busy_controller", run))):
        assert '"code":-32602' in out["busy"] and "Device or resource busy" in out["busy"], (kind, out)
        assert '"result":true' in out["last"], (kind, out)
        assert not out["socket_left"], kind


def test_vhost_user_reconnect_and_odd_masters(slaves):
    """a master that disappears mid-handshake, one that sends an unknown request, and a clean reconnect"""
    ours = slaves("ours", ["--control-only"])
    m = vu.Master(ours.sock("scsi0"))
    m.get_u64(vu.GET_FEATURES)
    m.close()                                           # gone without a word
    m = vu.Master(ours.sock("scsi0"))
    m.send(200, b"")                                    # >= VHOST_USER_MAX: the slave drops the connection
    with pytest.raises((ConnectionError, OSError)):
        m.s.settimeout(5)
        m.recv()
    m.close()
    m = vu.Master(ours.sock("scsi0"))
    assert m.set_u64(vu.SET_FEATURES, 1 << 40, need_reply=True) == 0      # unsupported feature bit: ignored, acked 0 like the reference
    assert m.get_u64(vu.GET_FEATURES) == 0x150000007
    m.close()
    # the RPC side is unaffected, and removing the controller removes its socket
    assert b'"result":true' in ours.call("remove_vhost_scsi_target", {"ctrlr": "scsi0", "scsi_target_num": 0})
    assert b'"result":true' in ours.call("remove_vhost_controller", {"ctrlr": "scsi0"})
    assert not os.path.exists(ours.sock("scsi0"))


def make_requests(seed, n=96):
    t = traces.fuzz_trace(n, NB, seed=seed, max_io_blocks=64, arena_bytes=16 << 20)
    a0 = np.zeros(t.arena_bytes, dtype=np.uint8)
    traces.fill_arena(a0, t)
    return vring.requests_from_trace(t, a0)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["kick", "poller", "kick-2gpus", "poller-2gpus"])
def test_cuda_vhost_user_io_matches_reference(slaves, mode):
    extra = ["--poller"] if mode.startswith("poller") else []
    if mode.endswith("2gpus"):
        # one controller, two GPUs: bdevs placed on the least-loaded GPU, the session's request queues dealt out over
        # both (queue r -> GPU r mod 2), every target reached from either GPU (own HBM or the peer's over NVLink)
        import torch
        if torch.cuda.device_count() < 2:
            pytest.skip("needs 2 GPUs (gpurun --gpus 2)")
        extra += ["--gpus", "0,1"]
    import json
    import re
    rq = make_requests(11)

    def iostat(s):
        """get_bdevs_iostat: what each bdev served, counted the way the bdev layer counts (the sessions are gone by
        now: the counters outlive them)"""
        time.sleep(0.5)
        return json.loads(re.sub(rb'"(tick_rate|\w+_latency_ticks)":\d+', rb'"\1":0', s.call("get_bdevs_iostat")))["result"]

    def ref_run(ref):
        lr, sr, img, rings = run_script(ref, rq, data=True)
        return {"log": lr, "mem": util.block_digests(mask(sr["end"], img, rings)).tolist(), "iostat": iostat(ref)}
    r = reference_side(slaves, "io", ref_run)                # the reference's side is the same for every mode
    skip_without_gpu_after_recording()
    ours = slaves("ours", extra)
    lo, so, img, rings = run_script(ours, rq, data=True)
    lr = transcript(r["log"])
    assert deliberate(lo) == deliberate(lr), f"protocol transcripts differ:\nours {lo}\nref  {lr}"
    assert_same_memory(mask(so["end"], img, rings), r["mem"])
    assert dict((k, v) for k, v in lo if v is not None)[vu.GET_VRING_BASE] is not None
    # the READ on queue 3 went to the hot-plugged target (a fresh Malloc bdev: zeros)
    data_off = META_END - 4 * 8192
    assert (so["end"][data_off:data_off + 4096] == 0).all()
    a, b = iostat(ours), r["iostat"]
    assert a == b, f"iostat differs:\nours {a}\nref  {b}"
    raw = [x for x in json.loads(ours.call("get_bdevs_iostat"))["result"] if x.get("name") == "M0"][0]
    assert raw["read_latency_ticks"] > 0 and raw["write_latency_ticks"] > 0, raw      # summed by the mover warps, 1 GHz ticks
    m0 = [x for x in a if x.get("name") == "M0"][0]
    assert m0["num_read_ops"] > 0 and m0["num_write_ops"] > 0 and [x for x in a if x.get("name") == "M1"][0]["num_read_ops"] == 1


class Vm:
    """a connected master with one request queue's worth of work laid out in its RAM"""

    def __init__(self, s: Slave, rq, seed):
        self.img = vring.build_image(rq, ring_size=256, seed=seed, mutate=False)
        self.ram = vu.GuestRam(self.img.arena.size)
        self.ram.mem[:] = self.img.arena
        self.rings = (small_ring(0), small_ring(1))
        for r in self.rings:
            self.ram.mem[r[0]:r[0] + 8192] = 0
        img = self.img
        self.queues = [vu.Queue(0, 16, *self.rings[0][:3]), vu.Queue(1, 16, *self.rings[1][:3]),
                       vu.Queue(2, img.ring_size, img.desc_off, img.avail_off, img.used_off)]
        self.m = vu.Master(s.sock("scsi0"))
        handshake(self.m, self.ram, img, self.queues)
        time.sleep(0.3)

    def io(self):
        self.queues[2].notify()
        self.queues[2].wait_used(self.ram, self.img.meta["placed"])
        c = self.img.masked(self.ram.mem)
        for used_off in [self.img.used_off] + [r[2] for r in self.rings]:
            c[used_off:used_off + 2] = 0
        return c

    def close(self, graceful=True):
        base = [self.m.get_vring_base(q.index) for q in self.queues] if graceful else None
        self.m.close()
        for q in self.queues:
            q.close()
        self.ram.close()
        return base


def two_vm_script(s: Slave):
    """VM A connects and idles; VM B connects, does I/O and disappears without a word; A then does its I/O and
    shuts down cleanly; a third VM re-uses the controller afterwards"""
    out = {}
    a = Vm(s, make_requests(21, 64), 3)
    b = Vm(s, make_requests(22, 64), 4)
    out["b"] = b.io()
    b.close(graceful=False)
    out["a"] = a.io()
    out["a_base"] = a.close()
    c = Vm(s, make_requests(23, 64), 5)
    out["c"] = c.io()
    out["c_base"] = c.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["kick", "poller"])
def test_cuda_vhost_user_sessions_come_and_go(slaves, mode):
    def ref_run(ref):
        out = two_vm_script(ref)
        return {**{k: util.block_digests(out[k]).tolist() for k in ("a", "b", "c")}, "a_base": out["a_base"], "c_base": out["c_base"]}
    want = reference_side(slaves, "sessions", ref_run)         # the reference's side is the same for both modes
    skip_without_gpu_after_recording()
    got = two_vm_script(slaves("ours", ["--poller"] if mode == "poller" else []))
    for k in ("a", "b", "c"):
        assert_same_memory(got[k], want[k], f"VM {k}: guest memory")
    assert got["a_base"] == want["a_base"] and got["c_base"] == want["c_base"]
    assert got["a_base"][2] == 64 - 0 or got["a_base"][2] > 0


def fuzz_script(m: vu.Master, ram: vu.GuestRam, rng, nmsg=60):
    """a random but reference-safe message sequence (queue indices allocated in order, GET_VRING_BASE only on
    allocated queues: the reference dereferences unallocated rings); everything else is fair game - unsupported
    feature bits, rings before memory, bad ring addresses, NOFD eventfds, REPLY_ACK on anything"""
    allocated = 0
    fds = []
    regs = [(0x100000000, ram.size, vu.UVA_BASE, 0, ram.fd)]

    def pick_index(may_allocate=True):
        nonlocal allocated
        if allocated == 0 or (may_allocate and allocated < 4 and rng.random() < 0.3):
            allocated += 1
            return allocated - 1
        return int(rng.integers(0, allocated))

    for _ in range(nmsg):
        k = int(rng.integers(0, 16))
        ack = bool(rng.integers(0, 2))
        if k == 0:
            m.get_u64(vu.GET_FEATURES)
        elif k == 1:
            m.get_u64(vu.GET_PROTOCOL_FEATURES)
        elif k == 2:
            m.get_u64(vu.GET_QUEUE_NUM)
        elif k == 3:
            f = int(rng.choice([0x154000007, 0x150000007, 0x100000000, 0x154000007 | 1 << 40, 0]))
            m.set_u64(vu.SET_FEATURES, f, need_reply=ack)
        elif k == 4:
            m.set_u64(vu.SET_PROTOCOL_FEATURES, int(rng.choice([0x9, 0x21f, 0x400, 0])), need_reply=ack)
        elif k == 5:
            m.set_mem_table(regs, need_reply=ack)
        elif k == 6:
            m.vring_state(vu.SET_VRING_NUM, pick_index(), int(rng.choice([16, 256])))
        elif k == 7:
            m.vring_state(vu.SET_VRING_BASE, pick_index(), int(rng.integers(0, 4)))
        elif k == 8:
            i = pick_index()
            base = vu.UVA_BASE + 65536 * i
            if rng.random() < 0.2:
                base = 0x1234000                              # not inside any region
            m.set_vring_addr(i, base, base + 8192, base + 4096)
        elif k in (9, 10):
            i = pick_index()
            req = vu.SET_VRING_KICK if k == 9 else vu.SET_VRING_CALL
            if rng.random() < 0.25:
                m.set_u64(req, i | vu.NOFD_MASK, need_reply=ack)
            else:
                fd = os.eventfd(0, os.EFD_NONBLOCK)
                fds.append(fd)
                m.set_u64(req, i, [fd], need_reply=ack)
        elif k == 11:
            m.vring_state(vu.SET_VRING_ENABLE, pick_index(), int(rng.integers(0, 2)))
        elif k == 12 and allocated:
            m.get_vring_base(pick_index(may_allocate=False))
        elif k == 13:
            m.get_config()
        elif k == 14:
            m.send(vu.SET_OWNER)
            m.log.append((vu.SET_OWNER, None))
        else:
            m.set_u64(vu.SET_CONFIG, 0, need_reply=True)
    for fd in fds:
        os.close(fd)


def test_vhost_user_random_message_sequences(slaves):
    """differential fuzzing of the protocol state machine: same random sequences, same replies"""
    def run(s):
        logs = []
        for seed in range(150):
            ram = vu.GuestRam(4 << 20)
            m = vu.Master(s.sock("scsi0"))
            try:
                fuzz_script(m, ram, np.random.default_rng(seed))
                logs.append(m.log)
            except (ConnectionError, OSError, TimeoutError) as e:
                logs.append(("dropped", type(e).__name__, len(m.log)))
            finally:
                m.close()
                ram.close()
            assert s.p.poll() is None, f"seed {seed}: the {s.kind} server died"
        return logs
    got = run(slaves("ours", ["--control-only"]))
    want = [transcript(x) for x in reference_side(slaves, "random_message_sequences", run)]
    assert len(got) == len(want) == 150
    for seed, (a, b) in enumerate(zip(got, want)):
        assert deliberate(a) == deliberate(b), f"seed {seed}: transcripts differ\nours {a}\nref  {b}"


def random_control_requests(ram, img, ring, rng):
    """8 control-queue requests of random type / subtype / target and random chain shape -> heads"""
    d = ram.mem[ring[0]:ring[0] + 16 * 16].view(vring.desc_dtype)
    heads = []
    for k in range(8):
        o = ring[3] + 64 * k
        typ = int(rng.choice([0, 0, 0, 1, 2, 9]))
        sub = int(rng.integers(0, 8))
        lun = bytes([int(rng.choice([1, 1, 1, 0])), int(rng.choice([0, 0, 1, 5, 9])), 0, int(rng.choice([0, 0, 1])), 0, 0, 0, 0])
        ram.mem[o:o + 24] = np.frombuffer(struct.pack("<II8sQ", typ, sub, lun, 0x2000 + k), np.uint8)
        ram.mem[o + 32:o + 48] = 0xEE
        shape = int(rng.integers(0, 8))
        req = (gpa_of(img, o), 24, 0)
        resp = (gpa_of(img, o + 32), int(rng.choice([1, 5, 5, 4, 0])), vring.F_WRITE)
        if shape == 0:
            req = (0x9_0000_0000, 24, 0)                                  # request unmapped
        elif shape == 1:
            resp = (0x9_0000_0000, resp[1], vring.F_WRITE)                # response unmapped
        chain = [req] if shape == 2 else [req, resp]                       # shape 2: no response descriptor
        s0 = 2 * k
        if shape == 3:                                                     # INDIRECT table
            tbl_off = o + 48 - (o + 48) % 16 + 16
            tbl = ram.mem[tbl_off:tbl_off + 32].view(vring.desc_dtype)
            for j, (a, ln, fl) in enumerate(chain):
                last = j + 1 == len(chain)
                tbl[j] = (a, ln, fl | (0 if last else vring.F_NEXT), 0 if last else j + 1)
            d[s0] = (gpa_of(img, tbl_off), 16 * len(chain), vring.F_INDIRECT, 0)
        else:
            for j, (a, ln, fl) in enumerate(chain):
                last = j + 1 == len(chain)
                nxt = 0 if last else s0 + j + 1
                if shape == 4 and not last:
                    nxt = 99                                               # next index beyond the table
                d[s0 + j] = (a, ln, fl | (0 if last else vring.F_NEXT), nxt)
        heads.append(s0 if shape != 5 else 16 + k)                          # shape 5: head beyond the ring
    return heads


def control_fuzz_script(s: Slave, seed: int):
    img = vring.build_image([], ring_size=256, seed=1, mutate=False)
    ram = vu.GuestRam(img.arena.size)
    ram.mem[:] = img.arena
    cq, eq = small_ring(0), small_ring(1)
    for r in (cq, eq):
        ram.mem[r[0]:r[0] + 8192] = 0
    queues = [vu.Queue(0, 16, *cq[:3]), vu.Queue(1, 16, *eq[:3]), vu.Queue(2, img.ring_size, img.desc_off, img.avail_off, img.used_off)]
    m = vu.Master(s.sock("scsi0"))
    try:
        handshake(m, ram, img, queues)
        time.sleep(0.25)
        publish(ram, cq, random_control_requests(ram, img, cq, np.random.default_rng(seed)))
        queues[0].notify()
        wait_used(ram, cq, 8)
        time.sleep(0.05)
        snap = ram.mem.copy()
        return mask(snap, img, (cq, eq)), used_set(snap, cq, 8)
    finally:
        m.close()
        for q in queues:
            q.close()
        ram.close()


def test_vhost_user_control_queue_fuzz(slaves):
    def ref_run(ref):
        out = []
        for seed in range(12):
            mem, used = control_fuzz_script(ref, seed)
            out.append({"mem": util.block_digests(mem).tolist(), "used": used})
        return out
    want = reference_side(slaves, "control_queue_fuzz", ref_run)
    ours = slaves("ours", ["--control-only"])
    for seed in range(12):
        a, ua = control_fuzz_script(ours, seed)
        ub = [tuple(u) for u in want[seed]["used"]]
        assert ua == ub, f"seed {seed}: used elements differ\nours {ua}\nref  {ub}"
        assert_same_memory(a, want[seed]["mem"], f"seed {seed}: guest memory")


def test_vhost_user_many_masters_and_hot_plug_at_once(slaves):
    """connections coming and going from several threads while targets are hot-plugged over RPC: the daemon
    must keep answering both (no crash, no stuck thread, no leaked listening socket)"""
    import threading
    ours = slaves("ours", ["--control-only"])
    errors = []

    def vm(k):
        try:
            for i in range(12):
                img = vring.build_image([], ring_size=64, seed=k * 100 + i, mutate=False, data_bytes=2 << 20)
                ram = vu.GuestRam(img.arena.size)
                ram.mem[:] = img.arena
                cq, eq = small_ring(0), small_ring(1)
                for r in (cq, eq):
                    ram.mem[r[0]:r[0] + 8192] = 0
                queues = [vu.Queue(0, 16, *cq[:3]), vu.Queue(1, 16, *eq[:3]), vu.Queue(2, 64, img.desc_off, img.avail_off, img.used_off)]
                m = vu.Master(ours.sock("scsi0"))
                handshake(m, ram, img, queues)
                if i % 3 == 0:
                    publish(ram, eq, event_buffers(ram, img, eq))
                    publish(ram, cq, control_requests(ram, img, cq))
                    queues[0].notify()
                    wait_used(ram, cq, 8)
                if i % 2:
                    for q in queues:
                        m.get_vring_base(q.index)
                m.close()                                  # every other one just disappears
                for q in queues:
                    q.close()
                ram.close()
        except Exception as e:                              # noqa: BLE001
            errors.append(f"vm {k}: {type(e).__name__}: {e}")

    threads = [threading.Thread(target=vm, args=(k,)) for k in range(6)]
    for t in threads:
        t.start()
    n = 0
    while any(t.is_alive() for t in threads):
        assert b'"result":1' in ours.call("add_vhost_scsi_lun", {"ctrlr": "scsi0", "scsi_target_num": 1, "bdev_name": "M1"})
        assert b'"result":true' in ours.call("remove_vhost_scsi_target", {"ctrlr": "scsi0", "scsi_target_num": 1})
        n += 1
    for t in threads:
        t.join()
    assert not errors, errors
    assert n > 0 and ours.p.poll() is None
    assert b'"scsi0"' in ours.call("get_vhost_controllers")
