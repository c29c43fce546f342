"""Static guards on the compiled lidar kernel (cuobjdump on the in-tree library; no GPU needed).

DESIGN.md section 3 rests on properties of the generated code that a harmless-looking source change can lose without any
test failing: the hot loop of the ray-march must contain no call (5 % of the kernel, DESIGN section 9) and no local-memory
traffic and stay short (it is the dependent chain of every lookup), and the kernel must fit the 40 registers that keep 12
CTAs of 128 threads resident per SM (32 for the 16-CTA variant)."""
import os
import re
import shutil
import subprocess

import pytest
from torch.utils.cpp_extension import CUDA_HOME

from f110_gymnasium_ros2_jazzy_b200 import _lib

CUOBJDUMP = shutil.which("cuobjdump") or (CUDA_HOME and shutil.which("cuobjdump", path=os.path.join(CUDA_HOME, "bin")))
pytestmark = pytest.mark.skipif(not CUOBJDUMP, reason="cuobjdump neither on PATH nor under CUDA_HOME")


def _functions(args):
    out = subprocess.check_output([CUOBJDUMP] + args + [_lib.LIB_PATH], stderr=subprocess.DEVNULL).decode()
    fns, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function\s*:?\s*(\S+)", line)
        if m:
            name = m.group(1).rstrip(":")
            fns[name] = []
        elif name is not None:
            fns[name].append(line)
    return fns


def _lidar_variants(fns):
    return {k: v for k, v in fns.items() if "lidar_kernel" in k}


def test_lidar_kernel_register_budget():
    fns = _lidar_variants(_functions(["-res-usage"]))
    assert len(fns) == 40                                       # fraction bits {generic, 19..22} x COUNT x MODE
    for name, lines in fns.items():
        text = " ".join(lines)
        reg = int(re.search(r"REG:(\d+)", text).group(1))
        local = int(re.search(r"LOCAL:(\d+)", text).group(1))
        assert reg <= 40, (name, reg)
        assert local <= 128, (name, local)                      # a few words of the per-unit bookkeeping, none in the hot loop


def test_lidar_hot_loop_has_no_call_and_no_local_memory():
    fns = _lidar_variants(_functions(["-sass"]))
    assert len(fns) == 40
    for name, lines in fns.items():
        ins = []
        for line in lines:
            m = re.search(r"/\*([0-9a-f]{4,5})\*/\s+(.*?);", line)
            if m:
                ins.append((int(m.group(1), 16), m.group(2)))
        loops = []
        for addr, text in ins:
            m = re.search(r"BRA\s+(?:P\d,\s*)?(?:`\(\.L_x_\d+\)|0x([0-9a-f]+))", text)
            if m and m.group(1) and int(m.group(1), 16) < addr:
                body = [t for a, t in ins if int(m.group(1), 16) <= a <= addr]
                if any("F2I.U32.F64" in t for t in body) and any("LDG" in t for t in body):
                    loops.append(body)
        assert loops, name
        hot = min(loops, key=len)                               # the guarded fixed-point march
        assert not any("CALL" in t for t in hot), name
        assert not any(("LDL" in t) or ("STL" in t) for t in hot), name
        tuned = "lidar_kernelILi0E" not in name
        lookups = sum("LDG" in t for t in hot)                  # the march is unrolled: two lookups per trip
        assert lookups in (1, 2), (name, lookups)
        per_lookup = len(hot) / lookups
        assert per_lookup <= (21 if tuned else 34), (name, len(hot), lookups)   # 19-20.5 tuned today (23 before the unroll, 38 with the world-frame march)
        if tuned:
            # no kernel parameter sits on the dependent chain of the tuned loop: at most the map base pointer is
            # rematerialised once per trip (issued at the top of the trip, consumed a whole lookup later)
            assert sum(("LDC" in t) or ("LDCU" in t) for t in hot) <= 1, name
