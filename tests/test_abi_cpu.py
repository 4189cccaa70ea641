"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol the
header declares, and fails loudly (no fallback) when no CUDA device exists."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest


def test_library_exports_every_declared_symbol():
    from bvh_b200 import capi

    names = capi.declared_symbols()
    assert len(names) >= 38
    L = capi.lib()
    for n in names:
        assert hasattr(L, n), n
    out = subprocess.run(["nm", "-D", "--defined-only", capi.SO_PATH], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert set(names) <= exported
    # nothing but the ABI leaks out of the shared object
    assert all(e.startswith("bvhgpu_") for e in exported), sorted(e for e in exported if not e.startswith("bvhgpu_"))[:5]


def test_pod_sizes_match_the_header():
    from bvh_b200 import dtypes as D

    hdr = open(os.path.join(os.path.dirname(os.path.dirname(__file__)), "include", "bvh_b200.h")).read()
    for name, size in (("bvh_aabb3f", 24), ("bvh_ray3f", 36), ("bvh_node3f", 64), ("bvh_flat3f", 36),
                       ("bvh_aabb3d", 48), ("bvh_ray3d", 72), ("bvh_node3d", 112), ("bvh_flat3d", 64)):
        assert name in hdr
    assert (D.AABB3F.itemsize, D.RAY3F.itemsize, D.NODE3F.itemsize, D.FLAT3F.itemsize) == (24, 36, 64, 36)
    assert (D.AABB3D.itemsize, D.RAY3D.itemsize, D.NODE3D.itemsize, D.FLAT3D.itemsize) == (48, 72, 112, 64)


def test_no_cpu_fallback_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from bvh_b200 import api, capi

    with pytest.raises(capi.BvhGpuError) as e:
        api.Context(0)
    assert e.value.status == capi.ERR_CUDA and "no CPU fallback" in str(e.value)


def test_library_contains_only_sm100a_code():
    import shutil

    from bvh_b200 import build, capi

    # the toolkit that built the library, which need not be on PATH
    cuobjdump = shutil.which("cuobjdump", path=os.path.dirname(build.NVCC) or None) or "cuobjdump"
    out = subprocess.run([cuobjdump, "--list-elf", capi.SO_PATH], capture_output=True, text=True).stdout
    archs = set(l.split(".")[-2] for l in out.splitlines() if ".cubin" in l)
    assert archs == {"sm_100a"}, archs


def test_product_never_imports_the_oracle():
    root = os.path.dirname(os.path.dirname(__file__))
    for dirpath, _, files in os.walk(os.path.join(root, "bvh_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("oracle/", "").lower() or f == "build.py", (dirpath, f)


def test_python_mirror_of_the_shard_macros_matches_the_header():
    """bvh_b200/capi.py restates BVHGPU_MAX_PEERS / BVHGPU_MAILBOX_BYTES / BVHGPU_SHARD_STAGE_BYTES and the struct bvhgpu_shard:
    compile the header's own macros with gcc and compare (a drift here would make ranks disagree about the staging layout)."""
    import ctypes as C
    import subprocess
    import tempfile

    from bvh_b200 import capi

    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "bvh_b200.h"
int main(void) {
    printf("%d %d %zu %zu", BVHGPU_MAX_PEERS, BVHGPU_MAILBOX_BYTES, sizeof(bvhgpu_shard), offsetof(bvhgpu_shard, shard_rays));
    size_t n[] = {0, 1, 2047, 2048, 1000000, 8000000, 16000000, 2147483647};
    for (int i = 0; i < 8; ++i) printf(" %zu", (size_t)BVHGPU_SHARD_STAGE_BYTES(n[i]));
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as d:
        c, exe = os.path.join(d, "m.c"), os.path.join(d, "m")
        open(c, "w").write(src)
        subprocess.run(["gcc", "-std=c11", "-I", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include"), c, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()
    vals = [int(x) for x in out]
    assert vals[0] == capi.MAX_PEERS and vals[1] == capi.MAILBOX_BYTES
    assert vals[2] == C.sizeof(capi.Shard) and vals[3] == capi.Shard.shard_rays.offset
    for n, want in zip((0, 1, 2047, 2048, 1000000, 8000000, 16000000, 2147483647), vals[4:]):
        assert capi.shard_stage_bytes(n) == want, n
