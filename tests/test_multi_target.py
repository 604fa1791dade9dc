"""One controller, several SCSI targets behind the same request queues (vhost_scsi.c:80-94, 361-387):
what OIM actually builds - MapVolume attaches every volume as another target of the one controller
(pkg/oim-controller/controller.go:55-156).

CPU: the restatement against the compiled reference.  GPU: the kernel against both, through a session with
a home target and through a controller-wide session; hot-plug while a session is open."""
import itertools

import numpy as np
import pytest

from oim_b200 import abi, traces, vring
from util import assert_cpls_equal, reference, sha

# target number -> blocks: different sizes so that one LBA is in range on some devices only
TARGETS = {1: 32768, 3: 4096, 6: 16384}
_seq = itertools.count()


def multi_trace(seed: int, n: int = 400, kind: str = "fuzz") -> traces.Trace:
    """a single-target trace re-addressed at random over the present targets and one absent slot"""
    if kind == "fuzz":
        t = traces.fuzz_trace(n, TARGETS[1], seed=seed, target=1, max_io_blocks=[8, 64, 300][seed % 3])
    else:
        t = traces.primary_trace(n, seed=seed, target=1)
    rng = np.random.default_rng(seed)
    pick = rng.choice([1, 3, 6, 5], size=len(t.reqs), p=[0.4, 0.3, 0.25, 0.05])
    ok = t.reqs["lun"][:, 0] == 1                      # leave the malformed addresses the fuzzer made alone
    t.reqs["lun"][ok, 1] = pick[ok].astype(np.uint8)
    return t


def run_oracle(cls, trace, names=None, ids=None):
    """-> cpls, arena, {target: store}, {target: scsi id}"""
    names = names or {}
    with cls(TARGETS[1], 512, 1, name=names.get(1), scsi_dev_id=(ids or {}).get(1)) as o:
        o.store[:] = traces.pattern_bytes(7, 0, o.store.size)
        for t in (3, 6):
            st = o.add_target(t, TARGETS[t], 512, name=names.get(t), scsi_dev_id=(ids or {}).get(t))
            st[:] = traces.pattern_bytes(7 + t, 0, st.size)
        arena = np.zeros(trace.arena_bytes, dtype=np.uint8)
        traces.fill_arena(arena, trace)
        cpls = o.submit(trace.reqs, trace.bind(arena.ctypes.data))
        stores = {1: o.store.copy(), 3: o.stores[3].copy(), 6: o.stores[6].copy()}
        sid = {t: o.target_scsi_dev_id(t) for t in TARGETS}
        return cpls, arena, stores, sid


@pytest.mark.parametrize("seed", range(700, 708))
@pytest.mark.parametrize("kind", ["fuzz", "primary"])
def test_multi_target_restatement_matches_reference(oracles, seed, kind):
    t = multi_trace(seed, kind=kind)
    names = {1: f"mt{seed}a", 3: f"mt{seed}b", 6: f"mt{seed}c"}

    def produce():
        c, a, s, i = run_oracle(oracles.RefOracle, t, names)
        return {"cpls": c, "arena_sha": sha(a), "store_sha": [sha(s[k]) for k in TARGETS], "ids": [i[k] for k in TARGETS]}
    want = reference("multi_target", f"{kind}{seed}", produce)
    wc, sid = want["cpls"], {k: int(x) for k, x in zip(TARGETS, want["ids"])}
    gc, ga, gs, _ = run_oracle(oracles.PortOracle, t, names, sid)
    assert_cpls_equal(gc, wc, t.reqs, "restatement vs reference")
    assert sha(ga) == str(want["arena_sha"])
    for k, w in zip(TARGETS, want["store_sha"]):
        assert sha(gs[k]) == str(w), f"store of target {k}"
    # every device took part, and the absent slot answered BAD_TARGET
    assert {int(x) for x in t.reqs["lun"][:, 1]} >= {1, 3, 5, 6}
    absent = (t.reqs["lun"][:, 0] == 1) & (t.reqs["lun"][:, 1] == 5) & (wc["resp_valid"] == 1)
    assert absent.any() and (wc["response"][absent] == abi.S_BAD_TARGET).all()


class Controller:
    """three Malloc bdevs on one controller, as MapVolume x3 leaves them"""

    def __init__(self, gpu, only=None):
        self.gpu = gpu
        tag = next(_seq)
        self.ctrlr = f"mtc{tag}"
        self.names = {t: f"mtb{tag}_{t}" for t in TARGETS}
        gpu.construct_vhost_scsi_controller(self.ctrlr)
        self.attached = set()
        for t in TARGETS:
            gpu.construct_malloc_bdev(TARGETS[t], 512, name=self.names[t], device=0)
            gpu.bdev_write_raw(self.names[t], 0, traces.pattern_bytes(7 + (t if t != 1 else 0), 0, TARGETS[t] * 512))
            if only is None or t in only:
                self.attach(t)

    def attach(self, t):
        self.gpu.add_vhost_scsi_lun(self.ctrlr, t, self.names[t])
        self.attached.add(t)

    def detach(self, t):
        self.gpu.remove_vhost_scsi_target(self.ctrlr, t)
        self.attached.discard(t)

    def ids(self):
        return {x["scsi_dev_num"]: x["id"] for x in self.gpu.get_vhost_controllers(self.ctrlr)[0]["backend_specific"]["scsi"]}

    def stores(self):
        return {t: self.gpu.bdev_read_raw(self.names[t], 0, TARGETS[t] * 512) for t in TARGETS}

    def close(self):
        for t in list(self.attached):
            self.detach(t)
        self.gpu.remove_vhost_controller(self.ctrlr)
        for t in TARGETS:
            self.gpu.delete_bdev(self.names[t])


def run_session(gpu, c, home, trace):
    import torch
    host_arena = np.zeros(trace.arena_bytes, dtype=np.uint8)
    traces.fill_arena(host_arena, trace)
    dev = torch.from_numpy(host_arena).to("cuda:0")
    torch.cuda.synchronize()
    with gpu.Lun(c.ctrlr, home, num_queues=1, queue_size=1024) as lun:
        cpls = lun.run(trace.reqs, trace.bind(dev.data_ptr()))
        torch.cuda.synchronize()
        stats = {t: lun.iostat(t) for t in TARGETS}
    return cpls, dev.cpu().numpy(), stats


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(720, 726))
@pytest.mark.parametrize("home", [1, 6, -1])
@pytest.mark.parametrize("kind", ["fuzz", "primary"])
def test_cuda_multi_target_matches_oracle(gpu, oracles, seed, home, kind):
    t = multi_trace(seed, kind=kind)
    c = Controller(gpu)
    try:
        checker = oracles.RefOracle if oracles.ref_available() and seed % 2 else oracles.PortOracle
        # INQUIRY reports bdev names and global SCSI device ids: give the checker ours where it can be told
        ids = c.ids()
        if checker is oracles.RefOracle and kind == "primary":
            checker = oracles.PortOracle           # the reference numbers its SCSI devices itself
        wc, wa, ws, _ = run_oracle(checker, t, c.names, ids)
        gc, ga, stats = run_session(gpu, c, home, t)
        assert_cpls_equal(gc, wc, t.reqs, f"cuda (home {home}) vs {checker.__name__}")
        assert (ga == wa).all(), f"client memory differs at {np.nonzero(ga != wa)[0][:8]}"
        gs = c.stores()
        for k in TARGETS:
            assert (gs[k] == ws[k]).all(), f"store of target {k}"
        # per-device counters: every good READ/WRITE is booked on the device it addressed
        good = (wc["resp_valid"] == 1) & (wc["response"] == abi.S_OK) & (wc["status"] == 0)
        for k in TARGETS:
            on_k = good & (t.reqs["lun"][:, 0] == 1) & (t.reqs["lun"][:, 1] == k) & ((t.reqs["lun"][:, 2] & 0x3f) == 0) & (t.reqs["lun"][:, 3] == 0)
            rd = np.isin(t.reqs["cdb"][:, 0], [0x08, 0x28, 0xa8, 0x88])
            wr = np.isin(t.reqs["cdb"][:, 0], [0x0a, 0x2a, 0xaa, 0x8a])
            moved = wc["data_transferred"] > 0
            assert stats[k]["num_read_ops"] >= int((on_k & rd & moved).sum())
            assert stats[k]["num_write_ops"] >= int((on_k & wr & moved).sum())
            if kind == "fuzz":
                assert stats[k]["num_read_ops"] + stats[k]["num_write_ops"] > 0
    finally:
        c.close()


def _rw(target, lba, nblk, write, addr):
    b = abi.Batch(target)
    (b.write if write else b.read)(lba, nblk, [(addr, nblk * 512)], tag=lba + 1)
    return b.arrays()


@pytest.mark.gpu
@pytest.mark.parametrize("poller", [False, True])
def test_cuda_hot_plug_into_open_session(gpu, poller):
    """add_vhost_scsi_lun / remove_vhost_scsi_target while a session is open (vhost_scsi.c:951-1100):
    the new device is reachable at once, the removed one answers BAD_TARGET, its bdev can be deleted"""
    import torch
    c = Controller(gpu, only={1})
    buf = torch.zeros(8192, dtype=torch.uint8).pin_memory()
    try:
        with gpu.Lun(c.ctrlr, -1, num_queues=1, queue_size=64) as lun:
            if poller:
                lun.start_poller(idle_timeout_ms=20000)
            run = lun.run                                     # doorbells when the poller is resident

            def io(target, lba, write=False):
                r, v = _rw(target, lba, 8, write, buf.data_ptr())
                return run(r, v)[0]

            assert io(3, 16)["response"] == abi.S_BAD_TARGET
            c.attach(3)                                       # hot-plug
            cp = io(3, 16)
            assert (cp["response"], cp["status"]) == (abi.S_OK, 0)
            assert (buf.numpy()[:4096] == traces.pattern_bytes(7 + 3, 16 * 512, 4096)).all()
            buf.numpy()[:4096] = 0xC3
            assert io(3, 24, write=True)["status"] == 0
            assert io(1, 16)["status"] == 0                    # the first device is still there
            c.detach(3)                                       # hot-unplug
            assert io(3, 16)["response"] == abi.S_BAD_TARGET
            gpu.delete_bdev(c.names[3])                       # no longer pinned by the session
            gpu.construct_malloc_bdev(TARGETS[3], 512, name=c.names[3], device=0)
            c.attach(6)
            assert io(6, 0)["status"] == 0
            # a second session on the same controller comes and goes while the first one stays resident
            with gpu.Lun(c.ctrlr, 6, num_queues=1, queue_size=64) as other:
                r, v = _rw(1, 8, 8, False, buf.data_ptr())
                assert other.run(r, v)[0]["status"] == 0
            assert io(1, 32)["status"] == 0
            if poller:
                assert lun.poller_running()
                lun.stop_poller()
    finally:
        c.close()


@pytest.mark.gpu
def test_cuda_multi_target_through_virtqueue(gpu, oracles):
    """the same through a guest virtio ring: descriptor walk, per-request target selection, responses"""
    import torch
    t = multi_trace(731, n=96)
    a0 = np.zeros(t.arena_bytes, dtype=np.uint8)
    traces.fill_arena(a0, t)
    rq = vring.requests_from_trace(t, a0)
    img = vring.build_image(rq, ring_size=1024, seed=9, mutate=False)
    assert img.meta["placed"] == len(rq)
    c = Controller(gpu)
    try:
        with oracles.PortOracle(TARGETS[1], 512, 1) as o:
            o.store[:] = traces.pattern_bytes(7, 0, o.store.size)
            for k in (3, 6):
                o.add_target(k, TARGETS[k])[:] = traces.pattern_bytes(7 + k, 0, TARGETS[k] * 512)
            ref_img = vring.build_image(rq, ring_size=1024, seed=9, mutate=False)
            n, la, lu = o.vq_process(ref_img)
            want_mem = ref_img.masked(ref_img.arena)
            want_stores = {1: o.store.copy(), 3: o.stores[3].copy(), 6: o.stores[6].copy()}
        dev = torch.from_numpy(img.arena).to("cuda:0")
        with gpu.Lun(c.ctrlr, -1, num_queues=1, queue_size=32) as lun:
            base = dev.data_ptr()
            lun.set_mem_table(img.region_table(base))
            lun.vq_attach(0, base + img.desc_off, base + img.avail_off, base + img.used_off, img.ring_size, 0, 0)
            assert lun.vq_kick() == 1
            lun.sync()
            assert lun.vq_detach(0) == (la, lu)
        got = img.masked(dev.cpu().numpy())
        assert (got == want_mem).all(), f"guest memory differs at {np.nonzero(got != want_mem)[0][:8]}"
        gs = c.stores()
        for k in TARGETS:
            assert (gs[k] == want_stores[k]).all()
    finally:
        c.close()
