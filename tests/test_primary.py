"""SURVEY.md 8(f) rank 1: the SPC primary commands a guest issues to attach the disk — INQUIRY (standard
and every VPD page), REPORT LUNS, MODE SENSE 6/10, MODE SELECT 6/10 (S/lib/scsi/scsi_bdev.c:188-1265,
1827-2077).  CPU: restatement vs the compiled reference + a golden fixture; GPU: the kernel vs both."""
import os

import numpy as np
import pytest

import util
from oim_b200 import abi, traces

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "primary.npz")
NB = 16384
NAME = "Malloc0"


def _one(o, cdb, n):
    buf = np.zeros(n, dtype=np.uint8)
    b = abi.Batch(0)
    b.add(np.array(list(cdb) + [0] * (32 - len(cdb)), dtype=np.uint8), abi.DIR_FROM_DEV, [(buf.ctypes.data, n)])
    return o.submit(*b.arrays())[0], buf


@pytest.mark.parametrize("which", ["port", "ref"])
def test_inquiry_known_answers(oracles, which):
    """what a Linux guest sees (pkg/oim-controller/controller_test.go:336-338 asserts vendor 'INTEL   ')"""
    cls = util.stored_reference("inquiry") if which == "ref" else oracles.PortOracle
    with cls(NB, name=NAME) as o:
        c, d = _one(o, [0x12, 0, 0, 0, 96], 96)
        assert c["status"] == 0 and c["resid"] == 0
        assert bytes(d[8:16]) == b"INTEL   " and bytes(d[16:32]) == b"Malloc disk     " and bytes(d[32:36]) == b"0001"
        assert d[0] == 0 and d[2] == 5 and d[4] == 91 and d[7] == 2
        c, d = _one(o, [0x12, 1, 0x80, 0, 64], 64)          # unit serial number = bdev name
        assert bytes(d[4:4 + len(NAME)]) == NAME.encode() and d[3] == len(NAME) + 1
        c, d = _one(o, [0x12, 1, 0xB0, 0, 64], 64)          # block limits: max transfer 4 MiB / 512
        assert int.from_bytes(bytes(d[8:12]), "big") == 8192 and int.from_bytes(bytes(d[24:28]), "big") == 256
        c, d = _one(o, [0x12, 1, 0xB2, 0, 64], 64)          # thin provisioning with UNMAP
        assert d[5] == 0x80 and d[6] == 2
        c, d = _one(o, [0xA0, 0, 0, 0, 0, 0, 0, 0, 0, 16], 16)      # REPORT LUNS: one LUN, id 0
        assert c["status"] == 0 and bytes(d) == bytes([0, 0, 0, 8] + [0] * 12)
        c, d = _one(o, [0x1A, 0, 0x08, 0, 64], 64)          # MODE SENSE(6) caching page: WCE set
        assert c["status"] == 0 and d[3] == 8 and d[12] == 0x08 and d[14] & 0x04
        c, d = _one(o, [0x1A, 0, 0xC8, 0, 64], 64)          # page control 3: saved values not supported
        assert c["status"] == 2 and c["sense"][12] == 0x39


@pytest.mark.parametrize("seed", range(500, 508))
def test_primary_restatement_matches_reference(oracles, seed):
    t = traces.primary_trace(300, seed=seed)

    def produce():
        with oracles.RefOracle(NB, name=NAME) as probe:
            dev_id = probe.scsi_dev_id
        cpls, arena, _ = util.run_oracle(oracles.RefOracle, t, NB, name=NAME)
        return {"cpls": cpls, "arena_sha": util.sha(arena), "scsi_dev_id": dev_id}
    want = util.reference("primary_commands", f"seed{seed}", produce)
    got = util.run_oracle(oracles.PortOracle, t, NB, name=NAME, scsi_dev_id=int(want["scsi_dev_id"]))
    util.assert_cpls_equal(got[0], want["cpls"], t.reqs, f"seed {seed}")
    assert util.sha(got[1]) == str(want["arena_sha"])


def test_primary_golden_fixture(oracles):
    """fixture produced by the reference (tests/golden/make_golden.py)"""
    z = np.load(GOLDEN)
    t = traces.primary_trace(int(z["n"]), seed=int(z["seed"]))
    assert (t.reqs.view(np.uint8) == z["reqs"].view(np.uint8)).all(), "trace generator drifted from the fixture"
    got = util.run_oracle(oracles.PortOracle, t, NB, name=NAME, scsi_dev_id=int(z["scsi_dev_id"]))
    util.assert_cpls_equal(got[0], z["cpls"], t.reqs)
    assert util.sha(got[1]) == str(z["arena_sha"])


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(520, 526))
def test_cuda_primary_commands(gpu, oracles, seed):
    t = traces.primary_trace(400, seed=seed)
    name = f"Malloc{seed}"
    want = util.run_oracle(oracles.PortOracle, t, NB, name=name, scsi_dev_id=0)
    got = util.run_cuda(gpu, t, NB, name=name, mem="device" if seed % 2 else "host")
    util.assert_cpls_equal(got[0], want[0], t.reqs, f"seed {seed}")
    assert (got[1] == want[1]).all(), f"response data differs at {np.nonzero(got[1] != want[1])[0][:8]}"
    if oracles.ref_available():
        with oracles.RefOracle(NB, name=name) as probe:
            dev_id = probe.scsi_dev_id
        if dev_id == 0:
            ref = util.run_oracle(oracles.RefOracle, t, NB, name=name)
            util.assert_cpls_equal(got[0], ref[0], t.reqs, f"seed {seed} vs reference")
            assert (got[1] == ref[1]).all()


@pytest.mark.gpu
def test_cuda_primary_golden_fixture(gpu):
    z = np.load(GOLDEN)
    t = traces.primary_trace(int(z["n"]), seed=int(z["seed"]))
    got = util.run_cuda(gpu, t, NB, name=NAME)
    if int(z["scsi_dev_id"]) == 0:
        util.assert_cpls_equal(got[0], z["cpls"], t.reqs)
        assert util.sha(got[1]) == str(z["arena_sha"])
