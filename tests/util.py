"""Helpers shared by the parity tests: run one trace through a checker or through the CUDA path, and the stored
results of the compiled reference that the tests compare against."""
from __future__ import annotations

import hashlib
import io
import itertools
import json
import lzma
import os

import numpy as np

from oim_b200 import abi, traces

_seq = itertools.count()

# What the compiled reference (oracle/_ref, built from the original project's sources) produced for the tests' cases.
# The tests compare against these files, so they run wherever the repository is, reference or not.  To regenerate them
# where oracle/_ref was built:  OIM_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"  and, for the reference's side
# of the GPU tests of the vhost-user transport,  OIM_RECORD_REFERENCE=1 python -m pytest tests/test_vhost_user.py -m gpu
# (without a GPU those record the reference's side and then skip).
REFERENCE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD = bool(os.environ.get("OIM_RECORD_REFERENCE"))


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def digest64(data: bytes) -> int:
    return int.from_bytes(hashlib.blake2b(data, digest_size=8).digest(), "little")


def block_digests(a: np.ndarray, block: int = 256 << 10) -> np.ndarray:
    """8-byte digest of every `block` bytes of `a` (the last block may be short): a compact record of a large buffer
    that still says where two buffers differ"""
    b = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    return np.array([digest64(b[o:o + block].tobytes()) for o in range(0, len(b), block)], dtype=np.uint64)


def assert_same_digests(got: np.ndarray, want: np.ndarray, what: str, block: int = 256 << 10):
    g = block_digests(got, block)
    assert len(g) == len(want), f"{what}: {len(g)} blocks, expected {len(want)}"
    bad = np.nonzero(g != want)[0]
    assert not len(bad), f"{what}: differs in {len(bad)} block(s) of {block} bytes, first at byte offset {int(bad[0]) * block}"


def _write_xz(path: str, data: bytes) -> None:
    os.makedirs(REFERENCE_DIR, exist_ok=True)
    with open(path, "wb") as f:
        f.write(lzma.compress(data, preset=9 | lzma.PRESET_EXTREME))


def reference(name: str, key: str, produce):
    """The reference's result for case `key` of `name`: a dict of numpy arrays stored in
    tests/golden/reference/<name>.npz.xz (an .npz, xz-compressed as a whole: the cases share most of their bytes).
    In record mode `produce()` runs the compiled reference and its result replaces the stored one."""
    path = os.path.join(REFERENCE_DIR, name + ".npz.xz")
    pre = key + "."
    stored = {}
    if os.path.exists(path):
        with lzma.open(path) as f, np.load(io.BytesIO(f.read())) as z:
            stored = {k: z[k] for k in z.files}
    if RECORD:
        out = {k: np.asarray(v) for k, v in produce().items()}
        stored = {k: v for k, v in stored.items() if not k.startswith(pre)}
        buf = io.BytesIO()
        np.savez(buf, **stored, **{pre + k: v for k, v in out.items()})
        _write_xz(path, buf.getvalue())
        return out
    out = {k[len(pre):]: v for k, v in stored.items() if k.startswith(pre)}
    assert out, f"{path}: no case {key} (see OIM_RECORD_REFERENCE in tests/util.py)"
    return out


def reference_json(name: str, key: str, produce):
    """The same for results that are JSON values (transcripts): tests/golden/reference/<name>.json.xz"""
    path = os.path.join(REFERENCE_DIR, name + ".json.xz")
    stored = {}
    if os.path.exists(path):
        with lzma.open(path, "rt") as f:
            stored = json.load(f)
    if RECORD:
        stored[key] = json.loads(json.dumps(produce()))
        _write_xz(path, json.dumps(stored, sort_keys=True, separators=(",", ":")).encode())
        return stored[key]
    assert key in stored, f"{path}: no case {key} (see OIM_RECORD_REFERENCE in tests/util.py)"
    return stored[key]


class StoredReference:
    """bindings.RefOracle as the known-answer tests drive it, from stored results (tests/golden/reference/known_answers.npz.xz):
    each submit() checks that the requests are the recorded ones, writes the bytes the reference left in the client
    buffers back into them and returns the reference's completions; with keep_store, `store` is the reference's backing
    store after that submit.  In record mode the live reference does the work and its results are written down."""

    def __init__(self, key: str, num_blocks: int, block_size: int = 512, target: int = 0, name: str | None = None,
                 keep_store: bool = False):
        self.key, self.calls, self.keep_store, self.live = key, itertools.count(), keep_store, None
        if RECORD:
            from oracle import bindings
            self.live = bindings.RefOracle(num_blocks, block_size, target, name=name)
            self.store = self.live.store
        else:
            self.store = np.zeros(num_blocks * block_size, dtype=np.uint8)

    def submit(self, reqs: np.ndarray, iovs: np.ndarray) -> np.ndarray:
        import ctypes as C
        bufs = [(int(a), int(n)) for a, n in zip(iovs["addr"], iovs["len"]) if a and n]

        def produce():
            cpls = self.live.submit(reqs, iovs)
            # the client buffers hold fill patterns of up to 4 MiB: stored as runs of equal bytes
            data = np.frombuffer(b"".join(C.string_at(a, n) for a, n in bufs), np.uint8)
            starts = np.r_[0, np.flatnonzero(np.diff(data)) + 1] if len(data) else np.zeros(0, np.int64)
            out = {"reqs": reqs, "cpls": cpls, "data": data[starts], "runs": np.diff(np.r_[starts, len(data)])}
            return {**out, "store": self.live.store.copy()} if self.keep_store else out
        r = reference("known_answers", f"{self.key}.{next(self.calls)}", produce)
        assert r["reqs"].tobytes() == np.ascontiguousarray(reqs).tobytes(), f"{self.key}: not the recorded requests"
        if not RECORD:
            data = np.repeat(r["data"], r["runs"])
            assert len(data) == sum(n for _, n in bufs), f"{self.key}: not the recorded client buffers"
            pos = 0
            for a, n in bufs:
                C.memmove(a, data[pos:pos + n].ctypes.data, n)
                pos += n
            if self.keep_store:
                self.store[:] = r["store"]
        return r["cpls"]

    def close(self):
        if self.live:
            self.live.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def stored_reference(name: str, **kw):
    """a stand-in for bindings.RefOracle within one test: its i-th instance replays case <name>.<i>"""
    n = itertools.count()
    return lambda *a, **k: StoredReference(f"{name}.{next(n)}", *a, **kw, **k)


def reference_run(name: str, key: str, trace: traces.Trace, num_blocks: int, **kw) -> dict:
    """run_oracle(RefOracle, ...) as stored: completions, SHA-256 of the client arena and of the backing store"""
    def produce():
        from oracle import bindings
        cpls, arena, store = run_oracle(bindings.RefOracle, trace, num_blocks, **kw)
        return {"cpls": cpls, "arena_sha": sha(arena), "store_sha": sha(store)}
    return reference(name, key, produce)


def run_oracle(cls, trace: traces.Trace, num_blocks: int, *, block_size: int = 512, store_seed: int | None = 7,
               arena_seed: int = 0x5EED, target: int = 0, removed: bool = False, name: str | None = None,
               scsi_dev_id: int | None = None):
    """-> (cpls, arena, store) after replaying `trace` on a CPU checker (RefOracle / PortOracle).
    name / scsi_dev_id: the identity INQUIRY reports (bdev name, global SCSI device id)."""
    o = cls(num_blocks, block_size, target, name=name, scsi_dev_id=scsi_dev_id)
    try:
        if store_seed is not None:
            o.store[:] = traces.pattern_bytes(store_seed, 0, o.store.size)
        if removed:
            o.set_removed(target, True)
        arena = np.zeros(trace.arena_bytes, dtype=np.uint8)
        traces.fill_arena(arena, trace, arena_seed)
        cpls = o.submit(trace.reqs, trace.bind(arena.ctypes.data))
        return cpls, arena, o.store.copy()
    finally:
        o.close()


def run_cuda(lib, trace: traces.Trace, num_blocks: int, *, block_size: int = 512, store_seed: int | None = 7,
             arena_seed: int = 0x5EED, target: int = 0, mem: str = "device", removed: bool = False,
             queue_size: int = 1024, name: str | None = None):
    """Same replay through liboimgpu.so on cuda:0.  mem="device": client buffers in HBM (a torch
    tensor); mem="host": client buffers in pinned, registered host memory."""
    import torch
    tag = next(_seq)
    bname, cname = name or f"par{tag}", f"parctl{tag}"
    lib.construct_malloc_bdev(num_blocks, block_size, name=bname, device=0)
    lib.construct_vhost_scsi_controller(cname)
    lib.add_vhost_scsi_lun(cname, target, bname)
    host_arena = np.zeros(trace.arena_bytes, dtype=np.uint8)
    traces.fill_arena(host_arena, trace, arena_seed)
    try:
        if store_seed is not None:
            lib.bdev_write_raw(bname, 0, traces.pattern_bytes(store_seed, 0, num_blocks * block_size))
        with lib.Lun(cname, target, num_queues=1, queue_size=queue_size) as lun:
            if removed:
                lun.set_removed(True)
            if mem == "device":
                dev = torch.from_numpy(host_arena).to("cuda:0")
                torch.cuda.synchronize()
                cpls = lun.run(trace.reqs, trace.bind(dev.data_ptr()))
                torch.cuda.synchronize()
                arena = dev.cpu().numpy()
            else:
                pinned = torch.from_numpy(host_arena.copy()).pin_memory()
                cpls = lun.run(trace.reqs, trace.bind(pinned.data_ptr()))
                arena = pinned.numpy().copy()
            stats = lun.iostat()
        store = lib.bdev_read_raw(bname, 0, num_blocks * block_size)
        return cpls, arena, store, stats
    finally:
        lib.remove_vhost_scsi_target(cname, target)
        lib.remove_vhost_controller(cname)
        lib.delete_bdev(bname)


def assert_cpls_equal(got: np.ndarray, want: np.ndarray, reqs: np.ndarray | None = None, what: str = ""):
    assert len(got) == len(want), f"{what}: {len(got)} completions, expected {len(want)}"
    for f in abi.CPL_PARITY_FIELDS:
        a, b = got[f].reshape(len(got), -1), want[f].reshape(len(want), -1)
        bad = np.nonzero((a != b).any(axis=1))[0]
        if len(bad):
            i = int(bad[0])
            extra = f"\nreq={reqs[i]}" if reqs is not None else ""
            raise AssertionError(f"{what}: completion field '{f}' differs at {len(bad)} requests, first #{i}: "
                                 f"got {got[i]} want {want[i]}{extra}")
