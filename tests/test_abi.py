"""The C-ABI boundary: wire layouts and exported symbols (no compute, runs without a GPU)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from oim_b200 import abi, build, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "oimgpu.h")


def _declared_functions() -> list[str]:
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(oimgpu_[a-z0-9_]+)\s*\(", src)))


def test_wire_struct_sizes_match_c(tmp_path):
    """numpy dtypes == C structs, checked by compiling a probe against include/oimgpu.h"""
    probe = tmp_path / "probe.c"
    probe.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "oimgpu.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
        "sizeof(struct oimgpu_req),sizeof(struct oimgpu_iov),sizeof(struct oimgpu_cpl),"
        "offsetof(struct oimgpu_req,tag),offsetof(struct oimgpu_req,cdb),offsetof(struct oimgpu_req,dir),"
        "offsetof(struct oimgpu_req,iovcnt),offsetof(struct oimgpu_req,iov_start),"
        "offsetof(struct oimgpu_cpl,sense),offsetof(struct oimgpu_cpl,used_len));return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(probe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [abi.req_dtype.itemsize, abi.iov_dtype.itemsize, abi.cpl_dtype.itemsize,
            abi.req_dtype.fields["tag"][1], abi.req_dtype.fields["cdb"][1], abi.req_dtype.fields["dir"][1],
            abi.req_dtype.fields["iovcnt"][1], abi.req_dtype.fields["iov_start"][1],
            abi.cpl_dtype.fields["sense"][1], abi.cpl_dtype.fields["used_len"][1]]
    assert got == want == [64, 16, 48, 8, 19, 51, 52, 56, 20, 40]


def test_request_prefix_is_virtio_scsi_cmd_req(tmp_path):
    """bytes 0..50 of oimgpu_req are struct virtio_scsi_cmd_req (linux/virtio_scsi.h)"""
    probe = tmp_path / "probe.c"
    probe.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include <linux/virtio_scsi.h>\n#include "oimgpu.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu\\n",sizeof(struct virtio_scsi_cmd_req),'
        "offsetof(struct virtio_scsi_cmd_req,tag),offsetof(struct virtio_scsi_cmd_req,cdb),"
        "sizeof(struct virtio_scsi_cmd_resp),offsetof(struct virtio_scsi_cmd_resp,status),"
        "offsetof(struct virtio_scsi_cmd_resp,sense));return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(probe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [51, abi.req_dtype.fields["tag"][1], abi.req_dtype.fields["cdb"][1], abi.RESP_SIZE,
                   abi.cpl_dtype.fields["status"][1] - 8, abi.cpl_dtype.fields["sense"][1] - 8]


def test_library_builds_loads_and_exports_every_declared_symbol():
    path = build.build()
    assert os.path.exists(path)
    declared = _declared_functions()
    assert len(declared) >= 35
    dll = C.CDLL(path)
    missing = [f for f in declared if not hasattr(dll, f)]
    assert not missing, f"declared in include/oimgpu.h but not exported: {missing}"
    bound = {name for name, _, _ in lib.SYMBOLS}
    assert set(declared) == bound, (set(declared) ^ bound)
    lib.load()      # types every entry point; still no compute
    assert lib.load().oimgpu_abi_version() == 1


def test_sm100a_sass_present():
    """the .so carries sm_100a code for our kernels (and nothing for another arch)"""
    path = build.build()
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", path], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out
    syms = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-symbols", path], capture_output=True, text=True).stdout
    for k in ("oim_lun_queue_kernel", "oim_copy_kernel", "oim_fill_kernel"):
        assert k in syms


def _cuda_device_present() -> bool:
    # (a device node name says nothing: a container may expose its GPU as /dev/nvidia3 alone)
    import torch
    return torch.cuda.is_available()


@pytest.mark.skipif(_cuda_device_present(), reason="only meaningful on a box without a GPU")
def test_no_cpu_fallback_without_gpu():
    """the product path fails loudly when there is no CUDA device"""
    with pytest.raises(lib.OimGpuError):
        lib.init([0])
    with pytest.raises(lib.OimGpuError):
        lib.construct_malloc_bdev(1024, 512)
