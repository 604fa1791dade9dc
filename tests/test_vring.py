"""Virtqueue level (SURVEY.md 8(a) a19-a22): real virtio split rings in a guest-memory image.
CPU: the C restatement against the compiled reference.  GPU: the kernel's own ring walk against both."""
import numpy as np
import pytest

import util
from oim_b200 import traces, vring


def make_requests(seed: int, n: int = 96, nb: int = 32768, contiguous: bool = False):
    t = traces.fuzz_trace(n, nb, seed=seed, max_io_blocks=[8, 64, 300][seed % 3], arena_bytes=16 << 20, contiguous=contiguous)
    a0 = np.zeros(t.arena_bytes, dtype=np.uint8)
    traces.fill_arena(a0, t)
    return vring.requests_from_trace(t, a0)


def run_kicks_oracle(cls, rq, nb, ring_size, seed, mutate=True, contiguous=False):
    """replay `rq` in as many kicks as the ring needs; -> [(masked image, sorted used entries, cursors)], store"""
    out = []
    with cls(nb) as o:
        o.store[:] = traces.pattern_bytes(7, 0, o.store.size)
        pos = kick = 0
        while pos < len(rq):
            img = vring.build_image(rq[pos:], ring_size=ring_size, seed=seed * 100 + kick, mutate=mutate, contiguous=contiguous)
            n, la, lu = o.vq_process(img)
            idx, ring = img.used_entries()
            out.append((img.masked(img.arena), sorted((int(i), int(l)) for i, l in ring[:idx]), (n, la, lu)))
            pos += img.meta["placed"]
            kick += 1
        return out, o.store.copy()


@pytest.mark.parametrize("seed", range(400, 412))
def test_vring_restatement_matches_reference(oracles, seed):
    nb, rq = 32768, make_requests(seed)
    ring = [64, 256, 1024][seed % 3]

    def produce():
        kicks, store = run_kicks_oracle(oracles.RefOracle, rq, nb, ring, seed)
        mem = [util.block_digests(m) for m, _, _ in kicks]
        return {"mem": np.concatenate(mem), "mem_count": np.array([len(m) for m in mem]),
                "cursors": np.array([c for _, _, c in kicks]),
                "used": np.array([u for _, used, _ in kicks for u in used], dtype=np.int64).reshape(-1, 2),
                "used_count": np.array([len(used) for _, used, _ in kicks]), "store_sha": util.sha(store)}
    want = util.reference("vring_kicks", f"seed{seed}", produce)
    got, got_store = run_kicks_oracle(oracles.PortOracle, rq, nb, ring, seed)
    assert len(got) == len(want["cursors"])
    used = np.split(want["used"], np.cumsum(want["used_count"])[:-1])
    mem = np.split(want["mem"], np.cumsum(want["mem_count"])[:-1])
    for k, (g, c, u, m) in enumerate(zip(got, want["cursors"], used, mem)):
        assert g[2] == tuple(int(x) for x in c), f"kick {k}: cursors"
        assert g[1] == [tuple(int(x) for x in e) for e in u], f"kick {k}: used elements"
        util.assert_same_digests(g[0], m, f"kick {k}: guest memory")
    assert util.sha(got_store) == str(want["store_sha"])


def test_vring_broken_avail_index(oracles):
    """avail->idx more than one ring ahead: 'the queue is unrecoverably broken' -> nothing is consumed"""
    rq = make_requests(5, n=8)
    for cls in ([oracles.PortOracle] + ([oracles.RefOracle] if oracles.ref_available() else [])):
        img = vring.build_image(rq, ring_size=64, seed=1, mutate=False)
        img.arena[img.avail_off + 2:img.avail_off + 4] = np.frombuffer(np.uint16(200).tobytes(), np.uint8)
        with cls(32768) as o:
            n, la, lu = o.vq_process(img)
        assert (n, la, lu) == (0, 0, 0) and img.used_entries()[0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("seed", list(range(420, 432)) + [1420, 1421, 1422, 1423])
@pytest.mark.parametrize("mem", ["device", "host"])
def test_cuda_vring_matches_oracle(gpu, oracles, seed, mem):
    """seeds >= 1000: every request's data descriptors are cuts of one guest buffer - the kernel moves a run of
    descriptors that continue each other as one segment, the reference copies them one by one"""
    import torch
    contiguous = seed >= 1000
    nb, rq = 32768, make_requests(seed, contiguous=contiguous)
    ring = [64, 256, 1024][seed % 3]
    checker = oracles.RefOracle if oracles.ref_available() and seed % 2 else oracles.PortOracle
    want, want_store = run_kicks_oracle(checker, rq, nb, ring, seed, contiguous=contiguous)

    gpu.construct_malloc_bdev(nb, 512, name=f"vq{seed}{mem}", device=0)
    gpu.construct_vhost_scsi_controller(f"vq{seed}{mem}.ctl")
    gpu.add_vhost_scsi_lun(f"vq{seed}{mem}.ctl", 0, f"vq{seed}{mem}")
    try:
        gpu.bdev_write_raw(f"vq{seed}{mem}", 0, traces.pattern_bytes(7, 0, nb * 512))
        with gpu.Lun(f"vq{seed}{mem}.ctl", 0, num_queues=2, queue_size=32) as lun:
            pos = kick = 0
            la = lu = 0
            while pos < len(rq):
                img = vring.build_image(rq[pos:], ring_size=ring, seed=seed * 100 + kick, contiguous=contiguous)
                # each kick is a fresh guest image (cursors restart at 0, as in the oracle replay)
                if mem == "device":
                    dev = torch.from_numpy(img.arena).to("cuda:0")
                else:
                    dev = torch.from_numpy(img.arena.copy()).pin_memory()
                base = dev.data_ptr()
                lun.set_mem_table(img.region_table(base))
                lun.vq_attach(1, base + img.desc_off, base + img.avail_off, base + img.used_off, img.ring_size, 0, 0)
                assert lun.vq_kick() == 1
                lun.sync()
                la, lu = lun.vq_detach(1)
                after = dev.cpu().numpy() if mem == "device" else dev.numpy().copy()
                idx, uring = img.used_entries(after)
                w = want[kick]
                assert (w[2][0], la, lu) == (w[2][0], w[2][1], w[2][2]), f"kick {kick}: cursors {la},{lu} vs {w[2]}"
                assert sorted((int(i), int(l)) for i, l in uring[:idx]) == w[1], f"kick {kick}: used elements"
                got = img.masked(after)
                assert (got == w[0]).all(), f"kick {kick}: guest memory differs at {np.nonzero(got != w[0])[0][:8]}"
                # the kernel publishes used elements in ring order
                assert [int(i) for i in uring[:idx]["id"]] == img.heads[:idx]
                pos += img.meta["placed"]
                kick += 1
        assert (gpu.bdev_read_raw(f"vq{seed}{mem}", 0, nb * 512) == want_store).all()
    finally:
        gpu.remove_vhost_scsi_target(f"vq{seed}{mem}.ctl", 0)
        gpu.remove_vhost_controller(f"vq{seed}{mem}.ctl")
        gpu.delete_bdev(f"vq{seed}{mem}")
