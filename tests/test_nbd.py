"""NBD export (SURVEY.md 8(f) rank 3; S/lib/nbd/nbd.c): the kernel's NBD transmission protocol - what /dev/nbdX
speaks to the daemon over the socketpair - served from the HBM-resident bdev.

No /dev/nbd* and no CAP_SYS_ADMIN exist in the build container or on the GPU box, so the test plays the kernel's
part itself: it keeps the "kernel" end of the socketpair and sends struct nbd_request / reads struct nbd_reply
(linux/nbd.h).  The reference's own server loop (nbd.c compiled into oracle/_ref, driven the same way) is the
checker: identical reply bytes, identical store.  The ioctl half of start_nbd_disk (NBD_SET_SOCK, NBD_DO_IT) is
covered only down to its error paths (tests/test_rpc_daemon.py)."""
import ctypes as C
import socket
import struct
import threading
import time

import numpy as np
import pytest

import util
from oim_b200 import traces

NB, BS = 8192, 512                     # 4 MiB
REQ_MAGIC, REP_MAGIC = 0x25609513, 0x67446698
READ, WRITE, DISC, FLUSH, TRIM = 0, 1, 2, 3, 4


def script(seed: int):
    """[(type, from, len, payload)] - aligned and misaligned I/O, out of range, flush, trim, an unknown command,
    a 1 MiB transfer; ends with a disconnect (even seeds) or a corrupt request (odd seeds)"""
    rng = np.random.default_rng(seed)
    ops = []
    for i in range(60):
        k = int(rng.integers(0, 12))
        frm = int(rng.integers(0, NB - 64)) * BS
        ln = int(rng.integers(1, 64)) * BS
        if k <= 3:
            ops.append((WRITE, frm, ln, traces.pattern_bytes(seed * 1000 + i, 0, ln).tobytes()))
        elif k <= 6:
            ops.append((READ, frm, ln, b""))
        elif k == 7:
            ops.append((TRIM, frm, ln, b""))
        elif k == 8:
            ops.append((FLUSH, 0, 0, b""))
        elif k == 9:
            bad = int(rng.integers(0, 5))
            if bad == 0:
                ops.append((READ, frm + 7, ln, b""))                              # offset not on a block
            elif bad == 1:
                ops.append((WRITE, frm, ln - 100, b"\x5a" * (ln - 100)))          # length not whole blocks
            elif bad == 2:
                ops.append((READ, NB * BS - BS, 4 * BS, b""))                     # runs off the end
            elif bad == 3:
                ops.append((TRIM, NB * BS, BS, b""))                              # starts at the end
            else:
                ops.append((TRIM, frm, 0, b""))                                   # "Can't unmap 0 bytes": EIO
        elif k == 10:
            ops.append((9, frm, ln, b""))                                         # unknown command: EIO, no payload
        else:
            ops.append((READ, 0, 1 << 20, b"") if i % 2 else (WRITE, 1 << 20, 1 << 20, traces.pattern_bytes(seed, 5, 1 << 20).tobytes()))
    return ops


def encode(op, handle: int) -> bytes:
    typ, frm, ln, payload = op
    return struct.pack(">II8sQI", REQ_MAGIC, typ, struct.pack("<Q", handle), frm, ln) + payload


def expect_len(op, reply: bytes) -> int:
    """bytes that follow the 16-byte reply header"""
    err = struct.unpack(">I", reply[4:8])[0]
    return op[2] if op[0] == READ and err == 0 else 0


def recv_exact(sock, n, pump):
    buf = b""
    t0 = time.time()
    while len(buf) < n:
        pump()
        try:
            chunk = sock.recv(n - len(buf))
            if chunk == b"":
                return buf + b"<closed>"
            buf += chunk
        except (BlockingIOError, socket.timeout):
            assert time.time() - t0 < 20, "no reply"
    return buf


def play(sock, ops, pump, tail: bytes):
    """the kernel's side: one request at a time; -> every byte the server sent, and whether it closed"""
    out = []
    for h, op in enumerate(ops):
        data = encode(op, 0x1000 + h)
        sent, t0 = 0, time.time()
        while sent < len(data):                       # big writes do not fit the socket buffer in one go
            try:
                sent += sock.send(data[sent:sent + 65536])
            except (BlockingIOError, socket.timeout):
                assert time.time() - t0 < 20, f"request {h} {op[:3]}: the server stopped reading"
            pump()
        hdr = recv_exact(sock, 16, pump)
        body = recv_exact(sock, expect_len(op, hdr), pump) if len(hdr) == 16 else b""
        out.append(hdr + body)
    sock.send(tail)
    out.append(recv_exact(sock, 1, pump))             # b"<closed>": the server hung up
    return out


def run_reference(oracles, ops, tail):
    """The reference's side lives on a thread of its own (SPDK state is thread-affine, and its transmit loop
    spins while the socket is full - it needs someone reading concurrently, as the kernel does); this thread
    plays the kernel."""
    a, b = socket.socketpair()
    a.settimeout(20)
    ready, stop, box = threading.Event(), threading.Event(), {}

    def server():
        o = oracles.RefOracle(NB, BS, 0, name=f"nbdref{abs(hash(tail)) % 1000}")
        try:
            o.store[:] = traces.pattern_bytes(7, 0, o.store.size)
            lib = o.lib
            lib.oimrefnbd_start.restype = C.c_void_p
            lib.oimrefnbd_start.argtypes = [C.c_char_p, C.c_int]
            lib.oimref_bdev_name.restype = C.c_char_p
            lib.oimref_bdev_name.argtypes = [C.c_void_p]
            box["started"] = bool(lib.oimrefnbd_start(lib.oimref_bdev_name(o.h), b.fileno()))
            ready.set()
            while not stop.is_set():
                lib.oimref_thread_poll(50)
            for _ in range(20):
                lib.oimref_thread_poll(50)
            box["store"] = o.store.copy()
        finally:
            ready.set()
            o.close()
    th = threading.Thread(target=server, daemon=True)
    th.start()
    assert ready.wait(20) and box.get("started")
    b.close()
    try:
        out = play(a, ops, lambda: None, tail)
    finally:
        stop.set()
        th.join(20)
        a.close()
    return out, box["store"]


def tails():
    return {"disc": encode((DISC, 0, 0, b""), 0xD15C), "garbage": b"\x00" * 28}


def reference_replies(oracles, key, ops, tail):
    """run_reference as stored: every reply (length, 8-byte digest, first 16 bytes) and the store's SHA-256"""
    def produce():
        out, store = run_reference(oracles, ops, tail)
        return {"len": [len(r) for r in out], "digest": np.array([util.digest64(r) for r in out], np.uint64),
                "head": np.array([np.frombuffer(r[:16].ljust(16, b"\0"), np.uint8) for r in out]), "store_sha": util.sha(store)}
    return util.reference("nbd_reference", key, produce)


def assert_replies_equal(ops, got, want):
    assert len(got) == len(want["len"])
    for i, g in enumerate(got):
        w = (int(want["len"][i]), int(want["digest"][i]))
        assert (len(g), util.digest64(g)) == w, \
            f"reply {i} to {ops[i][:3] if i < len(ops) else 'tail'} differs: {g[:24]!r} vs {bytes(want['head'][i])!r}..."


def test_reference_nbd_loop_known_answers(oracles):
    """the harness against the reference alone: known answers, so that the tests below compare against
    something that is itself pinned"""
    ops = [(WRITE, 4096, 1024, b"\xab" * 1024), (READ, 4096, 1024, b""), (READ, 4096 + 7, 512, b""), (TRIM, 4096, 512, b""),
           (READ, 4096, 1024, b""), (9, 0, 0, b""), (FLUSH, 0, 0, b"")]

    def produce():
        out, store = run_reference(oracles, ops, tails()["disc"])
        return {"replies": np.frombuffer(b"".join(out), np.uint8), "len": [len(r) for r in out], "store": store[4096:5120]}
    z = util.reference("nbd_known_answers", "disc", produce)
    out = [bytes(r) for r in np.split(z["replies"], np.cumsum(z["len"])[:-1])]
    store = np.zeros(8192, np.uint8)
    store[4096:5120] = z["store"]

    def rep(h, err):
        return struct.pack(">II8s", REP_MAGIC, err, struct.pack("<Q", 0x1000 + h))
    assert out[0] == rep(0, 0)
    assert out[1] == rep(1, 0) + b"\xab" * 1024
    assert out[2] == rep(2, 5)                                        # EIO, no payload
    assert out[3] == rep(3, 0)
    assert out[4] == rep(4, 0) + b"\x00" * 512 + b"\xab" * 512         # TRIM zero-filled the first block
    assert out[5] == rep(5, 5) and out[6] == rep(6, 0)
    assert out[7] == b"<closed>"
    assert (store[4096:4608] == 0).all() and (store[4608:5120] == 0xAB).all()


def run_restatement(oracles, ops, tail):
    """the C restatement (oracle/oim_oracle.c: oimorc_nbd_serve), blocking, on a thread of its own"""
    a, b = socket.socketpair()
    a.settimeout(20)
    o = oracles.PortOracle(NB, BS, 0)
    try:
        o.store[:] = traces.pattern_bytes(7, 0, o.store.size)
        o.lib.oimorc_nbd_serve.restype = C.c_int
        o.lib.oimorc_nbd_serve.argtypes = [C.c_void_p, C.c_int]
        rc = []

        def serve():
            rc.append(o.lib.oimorc_nbd_serve(o.h, b.fileno()))
            b.close()
        th = threading.Thread(target=serve, daemon=True)
        th.start()
        out = play(a, ops, lambda: None, tail)
        th.join(20)
        assert not th.is_alive()
        a.close()
        return out, o.store.copy(), rc[0]
    finally:
        o.close()


@pytest.mark.parametrize("seed", range(8))
def test_nbd_restatement_matches_reference(oracles, seed):
    ops = script(seed)
    tail = tails()["disc" if seed % 2 == 0 else "garbage"]
    want = reference_replies(oracles, f"seed{seed}", ops, tail)
    got, got_store, rc = run_restatement(oracles, ops, tail)
    assert rc == (0 if seed % 2 == 0 else -22)
    assert_replies_equal(ops, got, want)
    assert util.sha(got_store) == str(want["store_sha"])
    assert any(op[0] == TRIM and op[2] == 0 for s in range(8) for op in script(s)), "the zero-length TRIM case is in the scripts"


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
def test_cuda_nbd_matches_reference(gpu, oracles, seed):
    ops = script(seed)
    tail = tails()["disc" if seed % 2 == 0 else "garbage"]
    want = reference_replies(oracles, f"seed{seed}", ops, tail)
    name = f"nbd{seed}"
    gpu.construct_malloc_bdev(NB, BS, name=name, device=0)
    try:
        gpu.bdev_write_raw(name, 0, traces.pattern_bytes(7, 0, NB * BS))
        a, b = socket.socketpair()
        a.settimeout(20)
        rc = []
        def serve():
            rc.append(gpu.load().oimgpu_nbd_serve(name.encode(), b.fileno()))
            b.close()                                    # the caller owns the socket: the daemon closes it in nbd_stop
        th = threading.Thread(target=serve, daemon=True)
        th.start()
        got = play(a, ops, lambda: None, tail)
        th.join(20)
        assert not th.is_alive()
        a.close()
        assert rc == [0 if seed % 2 == 0 else -22]
        assert_replies_equal(ops, got, want)
        assert util.sha(gpu.bdev_read_raw(name, 0, NB * BS)) == str(want["store_sha"])
        st = gpu.get_bdevs_iostat(name)
        ok_reads = sum(1 for op, r in zip(ops, want["head"]) if op[0] == READ and not r[4:8].any())
        ok_writes = sum(1 for op, r in zip(ops, want["head"]) if op[0] == WRITE and not r[4:8].any())
        assert (st["num_read_ops"], st["num_write_ops"]) == (ok_reads, ok_writes)
    finally:
        gpu.delete_bdev(name)
