"""The C-ABI library loads and exports every symbol include/sihl_od.h declares (no compute calls: no GPU here)."""
import ctypes as C
import os
import re

from sihl_b200 import _native, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "sihl_od.h")).read()
    return sorted(set(re.findall(r"SIHL_OD_API\s+[\w\s\*]+?\b(sihl_od_\w+)\s*\(", text)))


def test_library_builds_and_loads():
    path = build.build()
    assert os.path.exists(path)
    lib = _native.load()
    assert lib.sihl_od_version() >= 100
    assert lib.sihl_od_last_error_string() is not None


def test_every_declared_symbol_is_exported_and_bound():
    declared = _declared()
    assert len(declared) >= 20
    lib = C.CDLL(build.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in sihl_od.h but not exported"
    assert sorted(_native.EXPORTED_SYMBOLS) == declared, "ctypes signatures and header disagree"


def test_library_reads_no_environment_variables():
    """Which kernel and grid an entry launches depends on its arguments alone, never on the process environment."""
    import shutil
    import subprocess

    import pytest
    nm = shutil.which("nm")
    if nm is None:
        pytest.skip("nm not found")
    path = build.build()
    out = subprocess.run([nm, "-D", "--undefined-only", path], capture_output=True, text=True, check=True).stdout
    imported = {line.split()[-1].split("@")[0] for line in out.splitlines() if line.strip()}
    assert not {name for name in imported if "getenv" in name}


def test_argument_errors_do_not_need_a_gpu():
    lib = _native.load()
    # n_levels out of range is rejected on the host, before any CUDA call
    rc = lib.sihl_od_anchors(None, 0, 640, 640, None, None, None, None)
    assert rc == 1
    assert b"level" in lib.sihl_od_last_error_string()
    rc = lib.sihl_od_topk(None, 1, 100, 5, None, None, None)
    assert rc == 1
    assert lib.sihl_od_nms_workspace_bytes(64, 256) == 0
    assert lib.sihl_od_nms_workspace_bytes(64, 8525) > 0


def test_sm100a_only_and_blackwell_bulk_copy_in_sass():
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        return
    out = subprocess.run([cuobjdump, "-lelf", build.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs
    sass = subprocess.run([cuobjdump, "-sass", build.LIB_PATH], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass and "SYNCS" in sass      # cp.async.bulk + mbarrier (TMA-class bulk copies)


def test_topk_and_nms_reject_cpu_tensors():
    import pytest
    import torch

    from sihl_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.topk_locations(torch.zeros(2, 300), 100)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.batched_nms(torch.zeros(10, 4), torch.zeros(10), torch.zeros(10, dtype=torch.int64), 0.5)


def test_exchange_and_split_helpers_without_a_gpu():
    """Size queries and argument checks of the multi-GPU exchange / class-split NMS entries are host-only."""
    lib = _native.load()
    assert lib.sihl_od_exchange_region_bytes(0) == 0 and lib.sihl_od_exchange_region_bytes(17) == 0
    assert lib.sihl_od_exchange_region_bytes(8) == 1280                # (18 * 8 + 1) words of 8 bytes, rounded to 256
    assert lib.sihl_od_exchange_region_bytes(1) == 256
    assert lib.sihl_od_nms_split_workspace_bytes(0, 100, 100) == 0
    small, big = lib.sihl_od_nms_split_workspace_bytes(1, 8525, 100), lib.sihl_od_nms_split_workspace_bytes(16, 34100, 100)
    assert 0 < small < big
    rc = lib.sihl_od_pos_loss_tiles_exchange(None, None, None, 1, 100, None, None, 10, 10, None, None, None, None, None, 0,
                                             None, None, None, None, 99, 0, None)
    assert rc == 1 and b"world" in lib.sihl_od_last_error_string()
    rc = lib.sihl_od_quad_matching(None, 10, None, None, 1, 5, 0, None, None, None, None, None, None, None, None)
    assert rc == 1 and b"topk" in lib.sihl_od_last_error_string()


def test_round2_entry_points_check_their_arguments_on_the_host():
    """Workspace queries and argument errors of the training-step, dtype-generic, wide-NMS and mAP entries need no GPU."""
    import ctypes as C
    lib = _native.load()
    # training step: workspace grows with the batch / gt capacity; too many images for the by-value gt layout; bad workspace
    a = lib.sihl_od_train_workspace_bytes(2, 2134, 27, 9)
    b = lib.sihl_od_train_workspace_bytes(64, 8525, 6400, 9)
    assert 0 < a < b and lib.sihl_od_train_workspace_bytes(2, 2134, 27, 0) == 0
    dummy = C.c_void_p(16)
    counts = (C.c_int32 * 600)(*([1] * 600))
    big = lib.sihl_od_train_workspace_bytes(600, 8525, 600, 9)
    rc = lib.sihl_od_train_assign(dummy, None, 8525, None, 0, 640, 640, dummy, counts, dummy, 600, 600, 9, dummy, dummy, dummy, 10,
                                  dummy, dummy, dummy, big, None)
    assert rc == 1 and b"gt_offsets on the device" in lib.sihl_od_last_error_string()
    rc = lib.sihl_od_train_assign(dummy, None, 8525, None, 0, 640, 640, dummy, None, dummy, 64, 6400, 9, dummy, dummy, dummy, 10,
                                  dummy, dummy, dummy, 16, None)
    assert rc == 1 and b"workspace too small" in lib.sihl_od_last_error_string()
    # map dtype codes: 0 / 1 / 2 only
    rc = lib.sihl_od_train_loss(dummy, None, None, None, 7, 1, 100, 0, dummy, dummy, None, 0, None, None, None, 0, 0, None, None,
                                dummy, dummy, None, None)
    assert rc == 1 and b"dtype" in lib.sihl_od_last_error_string()
    # the dense scan of half maps states its shape requirements (callers fall back to the candidate-first decode)
    rc = lib.sihl_od_dense_decode_t(dummy, dummy, dummy, 2, 1, 2134, 10, dummy, dummy, 320, 320, 0.05, dummy, 2134, dummy, dummy,
                                    dummy, 0, None)
    assert rc == 1 and b"C % 8" in lib.sihl_od_last_error_string()
    # stand-alone NMS: the whole-GPU path (and its mask workspace) from 8192 boxes, up to 90000
    small, wide, huge = (lib.sihl_od_batched_nms_workspace_bytes(n) for n in (8000, 30000, 100000))
    assert small == (2 * 8000 + 2) * 48 and wide > 30000 * 30000 // 8 and huge == (2 * 100000 + 2) * 48
    # N3: at most 1024 detections per image, 16 thresholds, 8 area ranges
    assert lib.sihl_od_map_workspace_bytes(100, 10, 4) == 100 * 10 * 4 * 4
    thr = (C.c_double * 10)(*[0.5 + 0.05 * i for i in range(10)])
    rc = lib.sihl_od_map_match(dummy, dummy, dummy, 1, 5000, None, None, dummy, 0, thr, 10, thr, 4, dummy, dummy, dummy, None,
                               dummy, None)
    assert rc == 1 and b"detections per image" in lib.sihl_od_last_error_string()
    assert lib.sihl_od_exchange_region_bytes(8) == 1280 and lib.sihl_od_exchange_barrier(None, 2, 0, None) == 1


def test_header_is_plain_c99():
    """include/sihl_od.h is the boundary a non-C++ host would bind: it must compile as C."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        return
    header = os.path.join(ROOT, "include", "sihl_od.h")
    res = subprocess.run([gcc, "-fsyntax-only", "-x", "c", "-std=c99", "-Wall", "-Werror", header], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr


def test_integration_stub_matches_the_abi():
    """The ctypes stub shown in INTEGRATION.md declares as many arguments as the library takes."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in ("sihl_od_assign_select", "sihl_od_assign_resolve"):
        m = re.search(r"_lib\." + name + r"\.argtypes = \[(.*?)\]", text, re.S)
        assert m, name
        n = len([x for x in m.group(1).replace("\n", " ").split(",") if x.strip()])
        assert n == len(_native._SIGNATURES[name][1]), (name, n)
