"""Boundary B1 (SURVEY.md 8(b)): the JSON-RPC wire behaviour of oim-gpu-vhost, compared reply by reply
with the REFERENCE'S OWN server (S/lib/jsonrpc + S/lib/rpc + the registered bdev / vhost handlers,
compiled into oracle/_ref; its replies stored in tests/golden/reference/rpc_transcripts.json.xz) and with the
expectations of OIM's Go tests (pkg/spdk/spdk_test.go:36-331, pkg/oim-controller/controller_test.go:226-304).

CPU: the daemon runs with --control-only (bookkeeping only, no data path exists in that mode).
GPU: the real daemon, plus a data check through the same process-external socket."""
import ctypes as C
import json
import os
import re
import socket
import subprocess
import sys
import time

import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DAEMON = os.environ.get("OIM_DAEMON_PATH") or os.path.join(ROOT, "oim_b200", "oim-gpu-vhost")   # override: sanitizer builds


class Client:
    """what pkg/spdk/client.go does: one JSON object per request, newline-terminated replies"""

    def __init__(self, path, pump=None):
        self.s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        t0 = time.time()
        while True:                      # the socket file appears at bind(), connections are taken from listen() on
            try:
                self.s.connect(path)
                break
            except (ConnectionRefusedError, FileNotFoundError):
                if time.time() - t0 > 10:
                    raise
                time.sleep(0.01)
        self.s.setblocking(False)
        self.pump = pump or (lambda: time.sleep(0.001))
        self.id = 0

    def raw(self, data: bytes, expect_reply=True, timeout=5.0) -> bytes:
        self.s.send(data)
        buf, t0 = b"", time.time()
        while time.time() - t0 < timeout:
            self.pump()
            try:
                chunk = self.s.recv(1 << 20)
                if chunk == b"":
                    return buf + b"<closed>"
                buf += chunk
                if buf.endswith(b"\n"):
                    return buf
            except BlockingIOError:
                if not expect_reply and time.time() - t0 > 0.15:
                    return buf
        return buf

    def call(self, method, params=None, **kw):
        self.id += 1
        req = {"jsonrpc": "2.0", "method": method, "id": self.id}
        if params is not None:
            req["params"] = params          # `params` omitted when nil (client.go:121-140)
        return self.raw((json.dumps(req) + "\n").encode(), **kw)


def norm(reply: bytes) -> str:
    s = reply.decode()
    s = re.sub(r'"tick_rate":\d+', '"tick_rate":"<hz>"', s)                          # the clock is the implementation's own
    return re.sub(r'"uuid":"(?!11111111-)[0-9a-f-]{36}"', '"uuid":"<uuid>"', s)     # random unless the test chose it


class Transcript:
    """The reference server's side of a test's conversation, as stored by util.reference_json: every request the test
    sent and the reference's reply, with the vhost socket directory written as <vdir>.  In record mode the requests go
    to the live reference server (`live`) and the transcript is written down."""

    def __init__(self, key: str, vdir: str, live: Client | None = None):
        self.key, self.vdir, self.live = key, vdir, live
        self.log = [] if live else util.reference_json("rpc_transcripts", key, None)
        self.pos = self.id = 0

    def raw(self, data: bytes, expect_reply=True, timeout=5.0) -> bytes:
        req = data.decode().replace(self.vdir, "<vdir>")
        if self.live:
            reply = self.live.raw(data, expect_reply, timeout)
            self.log.append([req, reply.decode().replace(self.vdir, "<vdir>")])
            return reply
        assert self.pos < len(self.log), f"{self.key}: the stored transcript ends before {req!r}"
        want, reply = self.log[self.pos]
        self.pos += 1
        assert req == want, f"{self.key}: the test sent {req!r} where the stored transcript has {want!r}"
        return reply.replace("<vdir>", self.vdir).encode()

    call = Client.call


@pytest.fixture()
def servers(oracles, sock_dir, request):
    """(ours, reference) clients sharing one vhost socket directory name: ours on a fresh server, the reference's
    replies from its stored transcript (recorded on a fresh reference server)"""
    from oim_b200 import build
    build.build()
    vdir = sock_dir / "vhost"
    vdir.mkdir()
    ours_sock, ref_sock = str(sock_dir / "ours.sock"), str(sock_dir / "ref.sock")
    mode = [] if os.environ.get("OIM_RPC_TEST_GPU") else ["--control-only"]
    procs = [subprocess.Popen([DAEMON, "-r", ours_sock, "-S", str(vdir), *mode], stderr=subprocess.PIPE)]
    if util.RECORD:
        # the reference server in a process of its own, so every test starts from SPDK's boot state
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "ref_rpc_server.py"), ref_sock, str(vdir)],
                                      stderr=subprocess.PIPE))
    for _ in range(500):
        if os.path.exists(ours_sock) and (not util.RECORD or os.path.exists(ref_sock)):
            break
        time.sleep(0.01)
    ref = Transcript(request.node.name, str(vdir), Client(ref_sock) if util.RECORD else None)
    try:
        yield Client(ours_sock), ref, str(vdir)
        if util.RECORD:
            util.reference_json("rpc_transcripts", ref.key, lambda: ref.log)
    finally:
        for p in procs:
            p.terminate()
            p.wait(5)


def both(servers, method, params=None):
    ours, ref, _ = servers
    a, b = norm(ours.call(method, params)), norm(ref.call(method, params))
    assert a == b, f"{method} {params}\n ours: {a}\n ref : {b}"
    return json.loads(a)


def test_rpc_transcript_matches_reference_server(servers):
    ours, ref, vdir = servers
    assert both(servers, "get_bdevs")["result"] == []
    assert both(servers, "get_bdevs", {"name": "no-such-bdev"})["error"]["code"] == -32602      # spdk_test.go:47-58
    assert both(servers, "get_vhost_controllers")["result"] == []
    # ---- Malloc bdevs (spdk_test.go:60-122)
    assert both(servers, "construct_malloc_bdev", {"num_blocks": 131072, "block_size": 512})["result"] == "Malloc0"
    assert both(servers, "construct_malloc_bdev", {"num_blocks": 2048, "block_size": 512, "name": "MyVol"})["result"] == "MyVol"
    assert both(servers, "construct_malloc_bdev", {"num_blocks": 2048, "block_size": 512})["result"] == "Malloc1"
    both(servers, "construct_malloc_bdev", {"num_blocks": 0, "block_size": 512})
    both(servers, "construct_malloc_bdev", {"num_blocks": 2048, "block_size": 512, "name": "MyVol"})      # duplicate
    both(servers, "construct_malloc_bdev", {"num_blocks": 2048, "block_size": 512, "uuid": "not-a-uuid"})
    both(servers, "construct_malloc_bdev", {"num_blocks": 2048, "block_size": 512, "name": "WithUuid",
                                            "uuid": "11111111-2222-3333-4444-555555555555"})
    both(servers, "construct_malloc_bdev", {"num_blocks": "8", "block_size": 512})                       # wrong type
    both(servers, "construct_malloc_bdev", {"num_blocks": 8, "block_size": 512, "bogus": 1})            # unknown key
    both(servers, "construct_malloc_bdev", {"block_size": 512})                                          # missing key
    both(servers, "construct_malloc_bdev")                                                               # no params
    r = both(servers, "get_bdevs", {"name": "WithUuid"})["result"][0]
    assert r["uuid"] == "11111111-2222-3333-4444-555555555555" and r["product_name"] == "Malloc disk"
    assert r["supported_io_types"] == {"read": True, "write": True, "unmap": True, "write_zeroes": True, "flush": True,
                                       "reset": True, "nvme_admin": False, "nvme_io": False}
    assert [b["name"] for b in both(servers, "get_bdevs")["result"]] == ["Malloc0", "MyVol", "Malloc1", "WithUuid"]
    both(servers, "get_bdevs", {"nam": "x"})
    # ---- vhost-scsi controllers (spdk_test.go:204-331)
    assert both(servers, "construct_vhost_scsi_controller", {"ctrlr": "vhost.0"})["result"] is True
    assert both(servers, "construct_vhost_scsi_controller", {"ctrlr": "vhost.0"})["error"]["message"] == "File exists"
    both(servers, "construct_vhost_scsi_controller", {"ctrlr": "vhost.1", "cpumask": "0x1"})
    both(servers, "construct_vhost_scsi_controller", {"ctrlr": "vhost.2", "cpumask": "0x4"})     # outside the app mask
    both(servers, "construct_vhost_scsi_controller", {"ctrlr": "vhost.2", "cpumask": "zz"})
    both(servers, "construct_vhost_scsi_controller", {})
    assert both(servers, "add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 0, "bdev_name": "Malloc0"})["result"] == 0
    assert both(servers, "add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 0, "bdev_name": "MyVol"})["error"]["message"] == "File exists"
    assert both(servers, "add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 8, "bdev_name": "MyVol"})["error"]["message"] == "Invalid argument"
    both(servers, "add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 2, "bdev_name": "missing"})
    assert both(servers, "add_vhost_scsi_lun", {"ctrlr": "nope", "scsi_target_num": 2, "bdev_name": "MyVol"})["error"]["message"] == "No such device"
    assert both(servers, "add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": -1, "bdev_name": "MyVol"})["result"] == 1
    # the controller may be named by its socket path (controller_test.go:179): the directory is stripped
    assert both(servers, "add_vhost_scsi_lun", {"ctrlr": vdir + "/vhost.1", "scsi_target_num": 7, "bdev_name": "Malloc1"})["result"] == 7
    both(servers, "add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 1.5, "bdev_name": "MyVol"})
    lst = both(servers, "get_vhost_controllers")["result"]
    assert [c["ctrlr"] for c in lst] == ["vhost.0", "vhost.1"] and lst[0]["cpumask"] == "0x1"
    assert lst[0]["socket"] == vdir + "/vhost.0" and lst[0]["iops_threshold"] == 60000
    assert lst[0]["backend_specific"]["scsi"][1] == {"scsi_dev_num": 1, "id": 1, "target_name": "Target 1",
                                                      "luns": [{"id": 0, "bdev_name": "MyVol"}]}
    both(servers, "get_vhost_controllers", {"name": "vhost.1"})
    assert both(servers, "get_vhost_controllers", {"name": "nope"})["error"]["code"] == -32603
    # ---- interrupt coalescing (vhost_rpc.c:493-544, vhost.c:358-381)
    assert both(servers, "set_vhost_controller_coalescing", {"ctrlr": "vhost.1", "delay_base_us": 50, "iops_threshold": 100000})["result"] is True
    assert both(servers, "set_vhost_controller_coalescing", {"ctrlr": "vhost.1", "delay_base_us": 50, "iops_threshold": 99})["error"]["message"] == "Invalid argument"
    assert both(servers, "set_vhost_controller_coalescing", {"ctrlr": "nope", "delay_base_us": 50, "iops_threshold": 100000})["error"]["message"] == "No such device"
    both(servers, "set_vhost_controller_coalescing", {"ctrlr": "vhost.1", "delay_base_us": 50})
    both(servers, "set_vhost_controller_coalescing", {"ctrlr": "vhost.1", "delay_base_us": -1, "iops_threshold": 100000})
    both(servers, "set_vhost_controller_coalescing", {"ctrlr": vdir + "/vhost.1", "delay_base_us": 0, "iops_threshold": 1000})
    c1 = both(servers, "get_vhost_controllers", {"name": "vhost.1"})["result"][0]
    assert (c1["delay_base_us"], c1["iops_threshold"]) == (0, 1000)
    both(servers, "set_vhost_controller_coalescing", {"ctrlr": "vhost.1", "delay_base_us": 25, "iops_threshold": 70000})
    # ---- get_bdevs_iostat (bdev_rpc.c:50-205): member names and order, one object per bdev in registration order
    st = both(servers, "get_bdevs_iostat")["result"]
    assert [x.get("name") for x in st[1:]] == ["Malloc0", "MyVol", "Malloc1", "WithUuid"] and "tick_rate" in st[0]
    assert list(st[1].keys()) == ["name", "bytes_read", "num_read_ops", "bytes_written", "num_write_ops", "bytes_unmapped",
                                  "num_unmap_ops", "read_latency_ticks", "write_latency_ticks", "unmap_latency_ticks"]
    assert len(both(servers, "get_bdevs_iostat", {"name": "MyVol"})["result"]) == 2
    assert both(servers, "get_bdevs_iostat", {"name": "nope"})["error"]["code"] == -32602
    both(servers, "get_bdevs_iostat", {"nam": "MyVol"})
    # ---- latency histogram (bdev_rpc.c:607-790): no I/O channel exists on either server here, so get returns the empty
    # histogram whether enabled or not (the per-channel -EFAULT needs a running session: tests/test_vhost_user.py)
    def hist(reply):
        return re.sub(r'"tsc_rate":\d+', '"tsc_rate":"<hz>"', reply)
    for m, pa in (("get_bdev_histogram", {"name": "MyVol"}), ("enable_bdev_histogram", {"name": "MyVol", "enable": True}),
                  ("get_bdev_histogram", {"name": "MyVol"}), ("enable_bdev_histogram", {"name": "MyVol", "enable": False}),
                  ("enable_bdev_histogram", {"name": "nope", "enable": True}), ("get_bdev_histogram", {"name": "nope"}),
                  ("enable_bdev_histogram", {"name": "MyVol"}), ("get_bdev_histogram", {})):
        a, b = hist(norm(ours.call(m, pa))), hist(norm(ref.call(m, pa)))
        assert a == b, f"{m} {pa}\n ours: {a[:300]}\n ref : {b[:300]}"
    import base64
    ref.call("get_bdev_histogram", {"name": "MyVol"})                    # (keeps the two clients' request ids in step)
    h = json.loads(ours.call("get_bdev_histogram", {"name": "MyVol"}))["result"]
    assert h["bucket_shift"] == 7 and len(base64.b64decode(h["histogram"])) == 58 * 128 * 8
    # ---- NBD export of OIM's local mode (nbd_rpc.c): no /dev/nbd* in the build container, so the error paths
    assert both(servers, "get_nbd_disks")["result"] == []
    assert both(servers, "start_nbd_disk", {"bdev_name": "MyVol", "nbd_device": "/dev/nbd-does-not-exist"})["error"]["code"] == -32602
    both(servers, "start_nbd_disk", {"bdev_name": "nope", "nbd_device": "/dev/null"})
    both(servers, "start_nbd_disk", {"bdev_name": "MyVol", "nbd_device": "/dev/null"})               # opens, but is no NBD device
    both(servers, "start_nbd_disk", {"bdev_name": "MyVol"})
    both(servers, "stop_nbd_disk", {"nbd_device": "/dev/nbd0"})
    both(servers, "get_nbd_disks", {"nbd_device": "/dev/nbd0"})
    # ---- teardown order of UnmapVolume (controller.go:159-212)
    assert both(servers, "remove_vhost_controller", {"ctrlr": "vhost.0"})["error"]["message"] == "Device or resource busy"
    assert both(servers, "remove_vhost_scsi_target", {"ctrlr": "vhost.0", "scsi_target_num": 0})["result"] is True
    both(servers, "remove_vhost_scsi_target", {"ctrlr": "vhost.0", "scsi_target_num": 0})
    both(servers, "remove_vhost_scsi_target", {"ctrlr": "vhost.0", "scsi_target_num": 9})
    both(servers, "remove_vhost_scsi_target", {"ctrlr": "nope", "scsi_target_num": 0})
    both(servers, "remove_vhost_scsi_target", {"ctrlr": "vhost.0", "scsi_target_num": 1})
    assert both(servers, "remove_vhost_controller", {"ctrlr": "vhost.0"})["result"] is True
    both(servers, "remove_vhost_controller", {"ctrlr": "vhost.0"})
    assert both(servers, "delete_bdev", {"name": "Malloc0"})["result"] is True
    both(servers, "delete_bdev", {"name": "Malloc0"})
    both(servers, "delete_bdev", {})
    both(servers, "get_bdevs")
    both(servers, "no_such_method", {"x": 1})


def test_rpc_framing_matches_reference_server(servers):
    ours, ref, _ = servers
    cases = [
        b'{"jsonrpc":"2.0","method":"get_bdevs","id":"abc"}\n',                       # string id echoed verbatim
        b'{"jsonrpc":"2.0","method":"get_bdevs","id":7,"extra":1}\n',                # unknown member -> invalid request
        b'{"jsonrpc":"1.0","method":"get_bdevs","id":7}\n',                          # wrong version
        b'{"method":"get_bdevs","id":8}\n',                                          # version is optional
        b'{"jsonrpc":"2.0","id":9}\n',                                               # no method
        b'{"jsonrpc":"2.0","method":5,"id":9}\n',
        b'{"jsonrpc":"2.0","method":"get_bdevs","params":5,"id":10}\n',              # params must be array/object
        b'{"jsonrpc":"2.0","method":"get_bdevs","params":[],"id":11}\n',             # positional params: decoder rejects
        b'[{"jsonrpc":"2.0","method":"get_bdevs","id":12}]\n',                       # batch: not supported
        b'  {"jsonrpc":"2.0",\n "method":"get_bdevs",\n "id":13}',                    # whitespace, no trailing newline
        b'{"jsonrpc":"2.0","method":"get_bdevs","id":14}{"jsonrpc":"2.0","method":"get_vhost_controllers","id":15}',
    ]
    for c in cases:
        a, b = norm(ours.raw(c)), norm(ref.raw(c))
        if c.count(b'"id"') == 2 and (a.count("\n") < 2 or b.count("\n") < 2):    # two requests in one write
            a, b = a + norm(ours.raw(b"", timeout=0.5)), b + norm(ref.raw(b"", timeout=0.5))
        assert a == b, f"{c!r}\n ours: {a}\n ref : {b}"
    # notification (no id): no reply at all; the connection stays usable
    for cl in (ours, ref):
        assert cl.raw(b'{"jsonrpc":"2.0","method":"get_bdevs"}\n', expect_reply=False) == b""
    assert norm(ours.call("get_bdevs")) .replace('"id":1', '"id":X') == norm(ref.call("get_bdevs")).replace('"id":1', '"id":X')
    # malformed JSON: no resync point in a JSON stream -> both servers drop the connection
    a, b = ours.raw(b'{"jsonrpc": nope}\n'), ref.raw(b'{"jsonrpc": nope}\n')
    assert a == b == b"<closed>"


def test_map_unmap_volume_sequence(servers):
    """the RPC sequence of oim-controller's ProvisionMallocBDev + MapVolume x2 + UnmapVolume
    (pkg/oim-controller/controller.go:55-256), replayed against both servers"""
    ours, ref, vdir = servers
    vol = "controller-test-volume"
    both(servers, "construct_vhost_scsi_controller", {"ctrlr": "scsi0"})     # test/pkg/spdk/spdk.go:204-226 creates by name
    assert both(servers, "get_bdevs", {"name": vol})["error"]["code"] == -32602          # CheckMallocBDev: absent
    assert both(servers, "construct_malloc_bdev", {"name": vol, "num_blocks": 64 * 2048, "block_size": 512})["result"] == vol
    for _ in range(2):                                                                   # MapVolume is idempotent
        assert both(servers, "get_bdevs", {"name": vol})["result"][0]["num_blocks"] == 131072
        ctrls = both(servers, "get_vhost_controllers")["result"]
        mapped = [(c["ctrlr"], t["scsi_dev_num"]) for c in ctrls for t in c["backend_specific"]["scsi"]
                  if t["luns"][0]["bdev_name"] == vol]
        if not mapped:
            for target in range(8):
                r = both(servers, "add_vhost_scsi_lun", {"ctrlr": vdir + "/scsi0", "scsi_target_num": target, "bdev_name": vol})
                if "result" in r:
                    mapped = [("scsi0", target)]
                    break
        assert mapped == [("scsi0", 0)]
    # UnmapVolume: find the target, remove it, leave the Malloc bdev alone (controller.go:202-209)
    assert both(servers, "remove_vhost_scsi_target", {"ctrlr": vdir + "/scsi0", "scsi_target_num": 0})["result"] is True
    assert both(servers, "get_bdevs", {"name": vol})["result"][0]["product_name"] == "Malloc disk"
    assert both(servers, "get_vhost_controllers")["result"][0]["backend_specific"]["scsi"] == []


@pytest.mark.gpu
def test_daemon_on_gpu_config1(sock_dir):
    """BASELINE config 1: 'Malloc bdev 64 MiB via oim-controller MapVolume' against the real daemon
    (HBM-backed stores): ProvisionMallocBDev -> MapVolume -> get -> UnmapVolume, plus the RBD-shaped volume
    of config 3 (construct_rbd_bdev as pkg/oim-controller/controller.go:284-295 issues it)."""
    from oim_b200 import build
    build.build()
    vdir = sock_dir / "vhost"
    vdir.mkdir()
    sock = str(sock_dir / "rpc.sock")
    proc = subprocess.Popen([DAEMON, "-r", sock, "-S", str(vdir), "-s", "256", "-R", "--gpus", "0", "--rbd-size", str(1 << 30)],
                            stderr=subprocess.PIPE)
    try:
        for _ in range(3000):
            if os.path.exists(sock):
                break
            time.sleep(0.01)
        c = Client(sock)

        def call(m, p=None):
            return json.loads(c.call(m, p, timeout=60))
        assert call("construct_vhost_scsi_controller", {"ctrlr": "scsi0"})["result"] is True
        assert call("construct_malloc_bdev", {"name": "vol-64m", "num_blocks": 131072, "block_size": 512})["result"] == "vol-64m"
        assert call("add_vhost_scsi_lun", {"ctrlr": str(vdir) + "/scsi0", "scsi_target_num": 0, "bdev_name": "vol-64m"})["result"] == 0
        r = call("construct_rbd_bdev", {"name": "pvc-1234", "block_size": 512, "pool_name": "rbd", "rbd_name": "pvc-1234",
                                        "user_id": "admin", "config": {"mon_host": "10.0.0.1:6789", "key": "AQ=="}})
        assert r["result"] == "pvc-1234"
        assert call("add_vhost_scsi_lun", {"ctrlr": "scsi0", "scsi_target_num": 1, "bdev_name": "pvc-1234"})["result"] == 1
        b = {x["name"]: x for x in call("get_bdevs")["result"]}
        assert b["vol-64m"]["product_name"] == "Malloc disk" and b["vol-64m"]["num_blocks"] == 131072
        assert b["pvc-1234"]["product_name"] == "Ceph Rbd Disk" and b["pvc-1234"]["num_blocks"] == (1 << 30) // 512
        scsi = call("get_vhost_controllers")["result"][0]["backend_specific"]["scsi"]
        assert [(t["scsi_dev_num"], t["luns"][0]["bdev_name"]) for t in scsi] == [(0, "vol-64m"), (1, "pvc-1234")]
        assert call("construct_rbd_bdev", {"block_size": 512, "rbd_name": "x"})["error"]["code"] == -32602   # pool_name missing
        for t in (0, 1):
            assert call("remove_vhost_scsi_target", {"ctrlr": "scsi0", "scsi_target_num": t})["result"] is True
        assert call("delete_bdev", {"name": "pvc-1234"})["result"] is True        # UnmapVolume deletes non-Malloc bdevs
        assert [x["name"] for x in call("get_bdevs")["result"]] == ["vol-64m"]
        assert call("get_nbd_disks")["result"] == []
        # no /dev/nbd0 on this box: whatever goes wrong in spdk_nbd_start is "Invalid parameters" (nbd_rpc.c:63-70)
        assert call("start_nbd_disk", {"bdev_name": "vol-64m", "nbd_device": "/dev/nbd0"})["error"]["code"] == -32602
    finally:
        proc.terminate()
        proc.wait(10)


def test_rpc_random_call_sequences(servers):
    """differential fuzzing of the bookkeeping: random create / attach / detach / delete / list sequences must
    produce identical replies (auto-naming counters, SCSI device ids, listing order, error messages)"""
    import random
    for seed in range(int(os.environ.get("OIM_RPC_FUZZ_SEEDS", "12"))):
        rng = random.Random(seed)
        bdevs = ["A", "B", "C", "Malloc0", "Malloc1", "gone"]
        ctrls = ["c0", "c1", "none"]
        for step in range(60):
            k = rng.randrange(11)
            if k == 0:
                p = {"num_blocks": rng.choice([2048, 4096, 0]), "block_size": rng.choice([512, 4096])}
                if rng.random() < 0.6:
                    p["name"] = rng.choice(bdevs[:3]) + f"_{seed}"
                both(servers, "construct_malloc_bdev", p)
            elif k == 1:
                both(servers, "delete_bdev", {"name": rng.choice(bdevs[:3]) + f"_{seed}" if rng.random() < 0.7 else rng.choice(bdevs)})
            elif k == 2:
                both(servers, "construct_vhost_scsi_controller", {"ctrlr": rng.choice(ctrls[:2]) + f".{seed}"})
            elif k == 3:
                both(servers, "remove_vhost_controller", {"ctrlr": rng.choice(ctrls) + f".{seed}"})
            elif k in (4, 5):
                both(servers, "add_vhost_scsi_lun", {"ctrlr": rng.choice(ctrls) + f".{seed}", "scsi_target_num": rng.choice([-1, 0, 1, 2, 7, 8]),
                                                     "bdev_name": rng.choice(bdevs[:3]) + f"_{seed}"})
            elif k == 6:
                both(servers, "remove_vhost_scsi_target", {"ctrlr": rng.choice(ctrls) + f".{seed}", "scsi_target_num": rng.choice([0, 1, 2, 7, 9])})
            elif k == 7:
                both(servers, "get_bdevs")
            elif k == 8:
                both(servers, "get_vhost_controllers")
            elif k == 9:
                both(servers, "get_bdevs", {"name": rng.choice(bdevs[:3]) + f"_{seed}"})
            else:
                both(servers, "get_bdevs_iostat")
        # leave both servers empty for the next seed (same calls on both, so they stay in step)
        for c in (f"c0.{seed}", f"c1.{seed}"):
            for t in range(8):
                both(servers, "remove_vhost_scsi_target", {"ctrlr": c, "scsi_target_num": t})
            both(servers, "remove_vhost_controller", {"ctrlr": c})
        for b in both(servers, "get_bdevs")["result"]:
            both(servers, "delete_bdev", {"name": b["name"]})


def test_config_dump_and_restore(sock_dir):
    """get_subsystems / get_subsystem_config + tools/oimcfg.py: the {method, params} lists of
    spdk_bdev_subsystem_config_json (S/lib/bdev/bdev.c:676-708; bdev_malloc.c:350-368, bdev_rbd.c:635-666) and
    spdk_vhost_config_json (S/lib/vhost/vhost.c:1460-1494; vhost_scsi.c:1459-1499), replayed into a fresh daemon"""
    from oim_b200 import build
    build.build()
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import oimcfg

    def daemon(tag):
        d = sock_dir / tag
        d.mkdir()
        (d / "vhost").mkdir()
        p = subprocess.Popen([DAEMON, "-r", str(d / "rpc.sock"), "-S", str(d / "vhost"), "--control-only"], stderr=subprocess.PIPE)
        for _ in range(500):
            if os.path.exists(d / "rpc.sock"):
                break
            time.sleep(0.01)
        return p, oimcfg.Rpc(str(d / "rpc.sock"))
    pa, a = daemon("a")
    pb, b = daemon("b")
    try:
        a.call("construct_malloc_bdev", {"num_blocks": 131072, "block_size": 512})
        a.call("construct_malloc_bdev", {"num_blocks": 4096, "block_size": 4096, "name": "Vol", "uuid": "11111111-2222-3333-4444-555555555555"})
        a.call("construct_rbd_bdev", {"block_size": 512, "pool_name": "rbd", "rbd_name": "pvc-1", "user_id": "admin", "name": "Rbd0"})
        a.call("construct_vhost_scsi_controller", {"ctrlr": "vhost.0"})
        a.call("construct_vhost_scsi_controller", {"ctrlr": "vhost.1", "cpumask": "0x1"})
        a.call("add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 0, "bdev_name": "Malloc0"})
        a.call("add_vhost_scsi_lun", {"ctrlr": "vhost.0", "scsi_target_num": 5, "bdev_name": "Rbd0"})
        a.call("set_vhost_controller_coalescing", {"ctrlr": "vhost.1", "delay_base_us": 40, "iops_threshold": 80000})
        assert [s["subsystem"] for s in a.call("get_subsystems")] == ["copy", "bdev", "scsi", "vhost"]
        bd = a.call("get_subsystem_config", {"name": "bdev"})
        assert bd[0] == {"method": "set_bdev_options", "params": {"bdev_io_pool_size": 65536, "bdev_io_cache_size": 256}}
        assert bd[2] == {"method": "construct_malloc_bdev", "params": {"name": "Vol", "num_blocks": 4096, "block_size": 4096,
                                                                       "uuid": "11111111-2222-3333-4444-555555555555"}}
        assert bd[3] == {"method": "construct_rbd_bdev", "params": {"name": "Rbd0", "pool_name": "rbd", "rbd_name": "pvc-1",
                                                                    "block_size": 512, "user_id": "admin"}}
        vh = a.call("get_subsystem_config", {"name": "vhost"})
        assert [x["method"] for x in vh] == ["construct_vhost_scsi_controller", "add_vhost_scsi_lun", "add_vhost_scsi_lun",
                                             "construct_vhost_scsi_controller", "set_vhost_controller_coalescing"]
        with pytest.raises(RuntimeError, match="Subsystem 'nope' not found"):
            a.call("get_subsystem_config", {"name": "nope"})
        cfg = oimcfg.save(a)
        assert oimcfg.load(b, json.loads(json.dumps(cfg))) == 8

        def strip(lst):                          # socket paths differ by directory
            return [{k: v for k, v in c.items() if k != "socket"} for c in lst]
        def bdevs(r):                            # construct_rbd_bdev carries no uuid (bdev_rbd.c:635-666): a restored RBD bdev gets a new one
            return [{k: (v if k != "uuid" or x["product_name"] != "Ceph Rbd Disk" else "<new>") for k, v in x.items()} for x in r.call("get_bdevs")]
        assert bdevs(a) == bdevs(b)
        assert strip(a.call("get_vhost_controllers")) == strip(b.call("get_vhost_controllers"))
        assert oimcfg.save(b) == cfg
    finally:
        for p in (pa, pb):
            p.terminate()
            p.wait(5)
