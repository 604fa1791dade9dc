"""The trace generators the parity tests and bench.py's SG legs rely on (host logic, CPU only)."""
import numpy as np

import util
from oim_b200 import traces, vring


def continues(iov):
    """mask over elements 1..: element j starts where element j-1 (non-empty) ended"""
    return (iov["len"][:-1] > 0) & (iov["addr"][:-1] + iov["len"][:-1] == iov["addr"][1:])


def test_sg_layouts_of_the_128k_legs():
    """bench.py seq128k_sg: same 33 element lengths, three placements in client memory"""
    n, io = 6, 131072
    for sg, shift in (("unaligned", 0), ("unaligned+3", 3), ("scattered", 0)):
        t = traces.uniform_trace(n, 1 << 16, io_blocks=256, pattern="seqwrite", sg=sg)
        k = len(t.iovs) // n
        assert k == 33
        for r in range(n):
            iov = t.iovs[r * k:(r + 1) * k]
            assert list(iov["len"]) == [100] + [4096] * 31 + [3996]
            base = r * t.meta["stride"] + shift
            # the elements tile the request's buffer exactly once
            spans = sorted((int(a), int(a + l)) for a, l in zip(iov["addr"], iov["len"]))
            assert spans[0][0] == base and spans[-1][1] == base + io
            assert all(a[1] == b[0] for a, b in zip(spans[:-1], spans[1:]))
            if sg == "scattered":
                assert not continues(iov).any(), "no element may continue its predecessor"
            else:
                assert continues(iov).all(), "one buffer cut at odd bytes: every element continues the one before"


def test_fuzz_traces_with_runs_of_contiguous_elements(oracles):
    """contiguous=True: multi-element SG lists are cuts of one client buffer; contiguous=False (the default, and the
    golden vectors' generator): never.  The restatement and the compiled reference agree on both."""
    nb = 16384
    plain = traces.fuzz_trace(300, nb, seed=11)
    runs = traces.fuzz_trace(300, nb, seed=11, contiguous=True)

    def joined(t):
        c = 0
        for r in t.reqs:
            iov = t.iovs[int(r["iov_start"]):int(r["iov_start"]) + int(r["iovcnt"])]
            if len(iov) > 1:
                real = iov[(iov["addr"] & traces.NULL_ADDR_FLAG) == 0]
                c += int(continues(real).sum()) if len(real) > 1 else 0
        return c
    # (the plain generator has a few contiguous lists too - its 512-byte page lists - so the golden vectors and every
    # fuzz test exercise joined runs; contiguous=True makes them the rule, at arbitrary byte cuts)
    assert joined(runs) > 2 * joined(plain) and joined(runs) > 300
    want = util.run_oracle(oracles.PortOracle, runs, nb)
    ref = util.reference_run("fuzz_runs", "seed11", runs, nb)
    util.assert_cpls_equal(want[0], ref["cpls"], runs.reqs, "runs")
    assert util.sha(want[1]) == str(ref["arena_sha"]) and util.sha(want[2]) == str(ref["store_sha"])
    assert (want[0]["status"] == 0).sum() > 200


def test_guest_images_with_runs_of_contiguous_descriptors():
    """vring.build_image(contiguous=True): a request's data descriptors continue each other in guest-physical memory"""
    t = traces.fuzz_trace(64, 32768, seed=1421, max_io_blocks=64, arena_bytes=16 << 20, contiguous=True)
    a0 = np.zeros(t.arena_bytes, dtype=np.uint8)
    traces.fill_arena(a0, t)
    rq = vring.requests_from_trace(t, a0)
    counts = {}
    for contiguous in (False, True):
        img = vring.build_image(rq, ring_size=256, seed=5, mutate=False, contiguous=contiguous)
        raw = img.arena[img.desc_off:img.desc_off + 16 * 256]
        addr, ln = raw.view("<u8")[0::2], raw.view("<u4")[2::4]
        spans = sorted((int(a), int(a) + int(l)) for a, l in zip(addr, ln) if l > 0)
        adj = sum(1 for x, y in zip(spans[:-1], spans[1:]) if x[1] == y[0])
        counts[contiguous] = adj
    # (request headers and response buffers are packed next to each other in both images: the difference is the data)
    assert counts[True] > counts[False] + 30, counts
