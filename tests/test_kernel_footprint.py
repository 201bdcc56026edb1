"""The top-K NMS shares SMs with the dense scan of the other steps in flight (csrc/od_nms.cu, file header).  The scan at
cfg1 runs two 256-thread CTAs per SM; a k_nms CTA must fit in what those two leave of the register file, and its
shared memory must stay small.  Checked on the built library with cuobjdump: no GPU needed."""
import os
import re
import shutil
import subprocess

import pytest

from sihl_b200 import _native, build

REGS_PER_SM = 65536
REG_ALLOC_UNIT = 256            # registers are allocated per warp in units of 256
SCAN_CTAS_PER_SM = 2            # od_infer.cu: 64-row stages, 2 CTAs per SM at cfg1
SCAN_THREADS = 256
NMS_SHARED_BUDGET = 64 * 1024   # static shared memory of a k_nms CTA (the top-K entry reserves no dynamic shared memory)
CFG1_SCAN = "_ZN4sihl18k_dense_decode_tmaILi5ELb1ELi64EfEEvNS_17DenseDecodeParamsEii"   # C = 80, fp32 maps


def _cuobjdump():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    return exe


def _res_usage():
    _native.load()                                   # builds the library if the tree changed
    out = subprocess.run([_cuobjdump(), "-res-usage", build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    usage = {}
    for name, regs, shared in re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:\d+ SHARED:(\d+)", out):
        usage[name] = (int(regs), int(shared))
    return usage


def _cta_registers(regs_per_thread, threads):
    per_warp = -(-regs_per_thread * 32 // REG_ALLOC_UNIT) * REG_ALLOC_UNIT
    return per_warp * (threads // 32)


def _topk_nms_threads():
    with open(os.path.join(build.CSRC, "od_nms.cu")) as fh:
        return int(re.search(r"constexpr int kNmsThreadsTopk = (\d+);", fh.read()).group(1))


def test_k_nms_fits_beside_two_scan_ctas():
    usage = _res_usage()
    threads = _topk_nms_threads()
    nms = usage[f"_ZN4sihl5k_nmsILi{threads}EEEvNS_9NmsParamsE"]        # k_nms<kNmsThreadsTopk>: the top-K entry
    scan_regs = _cta_registers(usage[CFG1_SCAN][0], SCAN_THREADS)
    assert _cta_registers(nms[0], threads) <= REGS_PER_SM - SCAN_CTAS_PER_SM * scan_regs, (nms, usage[CFG1_SCAN])
    assert nms[1] <= NMS_SHARED_BUDGET, nms


def test_top_k_workspace_covers_every_long_list():
    """Lists longer than the short-list body (256) run from the per-image workspace, not from dynamic shared memory."""
    lib = _native.load()
    assert lib.sihl_od_nms_workspace_bytes(64, 256) == 0
    assert lib.sihl_od_nms_workspace_bytes(1, 257) == 512 * 48
    assert lib.sihl_od_nms_workspace_bytes(64, 4096) == 64 * 4096 * 48
