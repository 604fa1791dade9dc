"""Pin the CPU checkers: restatement (oracle/oim_oracle.c) vs the compiled reference
(oracle/_ref, built from the original project's sources; its results stored under tests/golden/reference)
vs the committed golden vectors.  CPU only."""
import glob
import os

import numpy as np
import pytest

import util
from oim_b200 import abi, traces

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "fuzz_*.npz")))


def load_golden(path):
    z = np.load(path)
    t = traces.Trace(z["reqs"], z["iovs"], int(z["arena_bytes"]), os.path.basename(path))
    pay, pos = [], 0
    for o, l in zip(z["pay_off"], z["pay_len"]):
        pay.append((int(o), z["pay_data"][pos:pos + l]))
        pos += l
    t.meta["param_payloads"] = pay
    return t, z


def checkers(oracles):
    out = [oracles.PortOracle]
    if oracles.ref_available():
        out.append(oracles.RefOracle)
    return out


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_restatement_matches_golden_vectors(oracles, path):
    """golden vectors were produced by the reference itself (tests/golden/make_golden.py)"""
    t, z = load_golden(path)
    for cls in checkers(oracles):
        cpls, arena, store = util.run_oracle(cls, t, int(z["num_blocks"]), removed=bool(z["removed"]))
        util.assert_cpls_equal(cpls, z["cpls"], t.reqs, f"{cls.__name__}:{t.name}")
        assert util.sha(arena) == str(z["arena_sha"])
        assert util.sha(store) == str(z["store_sha"])


@pytest.mark.parametrize("seed", range(200, 212))
def test_restatement_matches_reference_on_fresh_fuzz(oracles, seed):
    nb = 32768
    t = traces.fuzz_trace(300, nb, seed=seed, max_io_blocks=[8, 64, 300][seed % 3])
    want = util.reference_run("fresh_fuzz", f"seed{seed}", t, nb)
    got = util.run_oracle(oracles.PortOracle, t, nb)
    util.assert_cpls_equal(got[0], want["cpls"], t.reqs, f"seed {seed}")
    assert util.sha(got[1]) == str(want["arena_sha"]) and util.sha(got[2]) == str(want["store_sha"])


# ---- known-answer cases of the reference's own unit tests ------------------------------------

def _one(o, cdb, direction, iovs):
    b = abi.Batch(0)
    b.add(cdb, direction, iovs)
    return o.submit(*b.arrays())[0]


@pytest.mark.parametrize("which", ["port", "ref"])
def test_scsi_bdev_ut_lba_range_and_xfer_len(oracles, which):
    """S/test/unit/lib/scsi/scsi_bdev.c/scsi_bdev_ut.c:639-794 (lba_range_test, xfer_len_test)"""
    cls = util.stored_reference("lba_range_and_xfer_len") if which == "ref" else oracles.PortOracle
    buf = np.zeros(5 * 512, dtype=np.uint8)
    with cls(4) as o:                                   # "Test block device size of 4 blocks"
        c = _one(o, abi.cdb_rw(abi.READ_16, 0, 1), abi.DIR_FROM_DEV, [(buf.ctypes.data, 512)])
        assert c["status"] == abi.STATUS_GOOD
        c = _one(o, abi.cdb_rw(abi.READ_16, 4, 1), abi.DIR_FROM_DEV, [(buf.ctypes.data, 512)])
        assert c["status"] == abi.STATUS_CHECK_CONDITION and c["sense"][12] == abi.ASC_LBA_OUT_OF_RANGE
        c = _one(o, abi.cdb_rw(abi.READ_16, 0, 4), abi.DIR_FROM_DEV, [(buf.ctypes.data, 4 * 512)])
        assert c["status"] == abi.STATUS_GOOD
        c = _one(o, abi.cdb_rw(abi.READ_16, 0, 5), abi.DIR_FROM_DEV, [(buf.ctypes.data, 5 * 512)])
        assert c["status"] == abi.STATUS_CHECK_CONDITION and c["sense"][12] == abi.ASC_LBA_OUT_OF_RANGE
    nb = 16400                                          # > 4 MiB / 512
    big = np.zeros(abi.MAX_XFER_BYTES + 512, dtype=np.uint8)
    with cls(nb) as o:
        c = _one(o, abi.cdb_rw(abi.READ_16, 0, 8192), abi.DIR_FROM_DEV, [(big.ctypes.data, abi.MAX_XFER_BYTES)])
        assert c["status"] == abi.STATUS_GOOD           # "max transfer length"
        c = _one(o, abi.cdb_rw(abi.READ_16, 0, 8193), abi.DIR_FROM_DEV, [(big.ctypes.data, abi.MAX_XFER_BYTES + 512)])
        assert c["status"] == abi.STATUS_CHECK_CONDITION
        assert c["sense"][2] & 0xF == abi.SK_ILLEGAL_REQUEST and c["sense"][12] == abi.ASC_INVALID_FIELD_IN_CDB
        c = _one(o, abi.cdb_rw(abi.READ_16, 0, 0), abi.DIR_FROM_DEV, [])
        assert c["status"] == abi.STATUS_GOOD and c["resid"] == 0     # "zero transfer length (valid)"
        c = _one(o, abi.cdb_rw(abi.READ_16, nb, 0), abi.DIR_FROM_DEV, [])
        assert c["status"] == abi.STATUS_CHECK_CONDITION and c["sense"][12] == abi.ASC_LBA_OUT_OF_RANGE


@pytest.mark.parametrize("which", ["port", "ref"])
def test_scsi_bdev_ut_xfer(oracles, which):
    """scsi_bdev_ut.c:796-897 (_xfer_test): READ16, WRITE16, UNMAP with 2 descriptors, SYNC16"""
    cls = util.stored_reference("xfer", keep_store=True) if which == "ref" else oracles.PortOracle
    with cls(2048) as o:
        o.store[:] = 0xEE
        buf = np.full(512, 0xA3, dtype=np.uint8)
        assert _one(o, abi.cdb_rw(abi.WRITE_16, 0, 1), abi.DIR_TO_DEV, [(buf.ctypes.data, 512)])["status"] == 0
        out = np.zeros(512, dtype=np.uint8)
        assert _one(o, abi.cdb_rw(abi.READ_16, 0, 1), abi.DIR_FROM_DEV, [(out.ctypes.data, 512)])["status"] == 0
        assert (out == 0xA3).all()
        pl = abi.unmap_param_list([(1, 2), (10, 3)])     # "Unmap 5 blocks using 2 descriptors"
        c = _one(o, abi.cdb_unmap(len(pl)), abi.DIR_TO_DEV, [(pl.ctypes.data, len(pl))])
        assert c["status"] == 0
        assert (o.store[512:3 * 512] == 0).all() and (o.store[10 * 512:13 * 512] == 0).all()
        assert (o.store[3 * 512:10 * 512] == 0xEE).all() and (o.store[13 * 512:14 * 512] == 0xEE).all()
        assert _one(o, abi.cdb_sync(abi.SYNCHRONIZE_CACHE_16, 0, 1), abi.DIR_FROM_DEV, [])["status"] == 0


@pytest.mark.parametrize("which", ["port", "ref"])
def test_vhost_ut_desc_to_iov(oracles, which):
    """S/test/unit/lib/vhost/vhost.c/vhost_ut.c:188-262: GPA->VVA and the 2 MiB / region split rule"""
    import ctypes as C
    import itertools
    regions = np.array([0, 0x400000, 0x1000000, 0x400000, 0x400000, 0x2000000], dtype=np.uint64)
    calls = itertools.count()

    def run(path, prefix, addr, length, start):
        fn = getattr(C.CDLL(path), prefix + "_desc_to_iov")
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32]
        out = np.zeros(4, dtype=abi.iov_dtype)
        n = fn(regions.ctypes.data, 2, addr, length, out.ctypes.data, start)
        return n, [(int(a), int(l)) for a, l in zip(out["addr"][:max(n, 0)], out["len"][:max(n, 0)])]

    def conv(addr, length, start=0):
        if which == "port":
            return run(oracles.PORT_SO, "oimorc", addr, length, start)
        n, iov = util.reference_json("known_answers", f"desc_to_iov.{next(calls)}",
                                     lambda: run(oracles.REF_SO, "oimref", addr, length, start))
        return n, [tuple(x) for x in iov]

    assert conv(0x110000, 0x1000) == (1, [(0x1110000, 0x1000)])
    assert conv(0x110000, 0x1000, abi.IOVS_MAX - 1) == (1, [(0x1110000, 0x1000)])
    assert conv(0x110000, 0x1000, abi.IOVS_MAX)[0] < 0
    assert conv(0x1F0000, 0x20000) == (1, [(0x11F0000, 0x20000)])         # 2 MiB boundary, same region
    assert conv(0x3F0000, 0x20000) == (2, [(0x13F0000, 0x10000), (0x2000000, 0x10000)])   # spans regions
    assert conv(0x900000, 0x1000)[0] < 0                                   # unmapped


# ---- bdevio data-integrity suite (S/test/bdev/bdevio/bdevio.c:388-800) on the checkers ----------

def bdevio_cases(nb):
    """(name, pattern, lba, nblocks, sg-lengths or None for write_zeroes(UNMAP), expect_ok)"""
    bs = 512
    return [
        ("write_read_512Bytes", 0xA3, 8, 1, [512], True),                      # :399
        ("write_read_4k", 0xA3, 8, 8, [4096], True),                           # :388 (offset 8192-ish)
        ("writev_readv_30x4k", 0xA3, 0, 240, [4096] * 30, True),               # :514
        ("writev_readv_size_gt_128k", 0xA3, 240, 264, [132 * 1024], True),     # :477
        ("writev_readv_size_gt_128k_two_iov", 0xA3, 240, 264, [128 * 1024, 4096], True),   # :494
        ("write_read_invalid_size", 0xA3, 8, 0, [0x1015], False),              # :536 not a multiple of the block size
        ("write_read_offset_plus_nbytes_equals_bdev_size", 0xA3, nb - 2, 2, [1024], True),  # :563
        ("write_read_offset_plus_nbytes_gt_bdev_size", 0xA3, nb - 1, 8, [4096], False),     # :593
        ("write_read_max_offset", 0xA3, 0xFFFFFFFFFFFFFFFF >> 9, 8, [4096], False),          # :618
        ("overlapped_write_read_8k_a", 0xA3, 0, 16, [8192], True),             # :642
        ("overlapped_write_read_8k_b", 0xBB, 8, 16, [8192], True),
    ]


class HostBuf:
    """client buffer in host memory (numpy)"""

    def __init__(self, n):
        self.a = np.zeros(max(n, 1), dtype=np.uint8)
        self.addr = self.a.ctypes.data

    def set(self, v):
        self.a[:len(v) if hasattr(v, "__len__") else None] = v

    def get(self):
        return self.a


@pytest.mark.parametrize("which", ["port", "ref"])
def test_bdevio_suite(oracles, which):
    cls = util.stored_reference("bdevio") if which == "ref" else oracles.PortOracle
    nb = 65536        # 32 MiB, as S/test/bdev/bdev.conf.in:5-7
    with cls(nb) as o:
        run_bdevio(o.submit, HostBuf, nb)


def run_bdevio(submit, alloc, nb):
    """write pattern -> read back -> compare, as blockdev_write_read (bdevio.c:334-386).
    `alloc(n)` returns a client buffer with .addr / .set(value) / .get() -> numpy."""
    for name, pat, lba, nblk, lens, ok in bdevio_cases(nb):
        total = sum(lens)
        tx, rx = alloc(total), alloc(total)
        tx.set(pat)

        def sg(base):
            return [(base + sum(lens[:k]), lens[k]) for k in range(len(lens))]
        use16 = lba >= 1 << 32 or nblk >= 1 << 16
        b = abi.Batch(0)
        b.write(lba, max(nblk, 1), sg(tx.addr), opcode=abi.WRITE_16 if use16 else abi.WRITE_10)
        b.read(lba, max(nblk, 1), sg(rx.addr), opcode=abi.READ_16 if use16 else abi.READ_10)
        c = submit(*b.arrays())
        if ok:
            assert (c["status"] == 0).all(), name
            assert (rx.get()[:total] == pat).all(), name
        else:
            assert (c["status"] == abi.STATUS_CHECK_CONDITION).all(), name
    # write_zeroes 4K / 1M / 3M / 3.5M (bdevio.c:700-800) through UNMAP, the Malloc module's fill path
    for nbytes in (4096, 1 << 20, 3 << 20, 3 << 20 | 1 << 19):
        blocks = nbytes // 512
        tx = alloc(min(nbytes, abi.MAX_XFER_BYTES))
        tx.set(0xA3)
        b = abi.Batch(0)
        done = 0
        while done < blocks:                       # pre-fill with the pattern, <= 4 MiB per WRITE
            n = min(blocks - done, abi.MAX_XFER_BYTES // 512)
            b.write(done, n, [(tx.addr, n * 512)], opcode=abi.WRITE_16)
            done += n
        pl = abi.unmap_param_list([(0, blocks)])
        plbuf = alloc(len(pl))
        plbuf.set(pl)
        b.add(abi.cdb_unmap(len(pl)), abi.DIR_TO_DEV, [(plbuf.addr, len(pl))])
        rx = alloc(min(nbytes, abi.MAX_XFER_BYTES))
        rx.set(0x55)
        n = min(blocks, abi.MAX_XFER_BYTES // 512)
        b.read(blocks - n, n, [(rx.addr, n * 512)], opcode=abi.READ_16)
        c = submit(*b.arrays())
        assert (c["status"] == 0).all(), nbytes
        assert (rx.get()[:n * 512] == 0).all(), nbytes
