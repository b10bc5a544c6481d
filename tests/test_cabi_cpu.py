"""CPU: the C-ABI library builds, loads, exports every symbol include/robotick.h declares,
and fails loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import re

import numpy as np

import pytest

import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, build, layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return rk.load()


def _declared_symbols():
    syms = set()
    for hdr in os.listdir(os.path.join(ROOT, "include")):
        if not hdr.endswith(".h"):
            continue
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        syms |= set(re.findall(r"\b(rk_[a-z0-9_]+)\s*\(", text))
    return syms


def test_exports_every_declared_symbol(lib):
    syms = _declared_symbols()
    assert len(syms) >= 25
    for s in sorted(syms):
        assert hasattr(lib, s), f"librobotick_b200.so does not export {s}"


def test_version_and_layout(lib):
    assert lib.rk_version() == 100
    assert lib.rk_vdt_state_words() == layout.VS_WORDS == 112
    assert lib.rk_vdt_state_bytes(10) == 10 * 448


def test_default_params_match(lib):
    p = _cabi.VdtParams()
    lib.rk_vdt_default_params(C.byref(p))
    assert bytes(p) == bytes(rk.default_params())


def test_arm_abi(lib):
    p = _cabi.AdtParams()
    lib.rk_adt_default_params(C.byref(p))
    assert bytes(p) == bytes(_cabi.default_arm_params())
    assert lib.rk_adt_state_words() == layout.AS_WORDS == 76
    assert lib.rk_adt_state_bytes(3) == 3 * 304 and lib.rk_adt_cmdtab_bytes(2) == 2 * 4160
    assert C.sizeof(_cabi.AdtPosCmdSeq) == 776  # sizeof(ADTModePositioningSeq::PosCmdSeq), SURVEY 8a
    text = open(os.path.join(ROOT, "include", "robotick.h")).read()
    for name, val in (("RK_AS_JOINT0", layout.AS_JOINT0), ("RK_AS_JFLAGS", layout.AS_JFLAGS), ("RK_AS_MG_TX", layout.AS_MG_TX),
                      ("RK_AS_BLDC_TX0", layout.AS_BLDC_TX0), ("RK_AS_WORDS", layout.AS_WORDS)):
        assert re.search(rf"{name}\s*=\s*{val}\b", text), name
    import torch

    if not torch.cuda.is_available():
        h = C.c_void_p()
        assert lib.rk_adt_create(C.byref(h), None) == 2  # RK_ERR_CUDA: no CPU fallback
        buf = (C.c_uint32 * 2048)()
        addr = (C.addressof(buf) + 15) & ~15
        assert lib.rk_adt_update(C.byref(p), C.c_void_p(addr), C.c_void_p(addr), 1, 1, None, None) == 2
    assert lib.rk_adt_update(C.byref(p), C.c_void_p(8), C.c_void_p(16), 1, 1, None, None) == 1


def test_header_enums_match_python_layout():
    text = open(os.path.join(ROOT, "include", "robotick.h")).read()
    assert "RK_VS_INTERP0 = 12" in text
    assert layout.VS_CTRL0 == 48 and layout.VS_MOTOR0 == 80


def test_new_block_layouts_match_header(lib):
    text = open(os.path.join(ROOT, "include", "robotick.h")).read()
    for name, val in (("RK_IP_FLAGS", layout.IP_FLAGS), ("RK_IP_SREG", layout.IP_SREG), ("RK_IP_WORDS", layout.IP_WORDS),
                      ("RK_HS_WAIT_CNT", None), ("RK_HS_VEL_DIR", layout.HS_VEL_DIR), ("RK_HS_WORDS", layout.HS_WORDS),
                      ("RK_RS_NO_CMD_CNT", layout.RS_NO_CMD_CNT), ("RK_RS_ABORT", layout.RS_ABORT), ("RK_RS_WORDS", layout.RS_WORDS),
                      ("RK_RI_FLOOR", layout.RI_FLOOR), ("RK_RI_WORDS", layout.RI_WORDS), ("RK_RI_X", layout.RI_X)):
        if val is None:
            assert name in text
        else:
            assert re.search(rf"{name}\s*=\s*{val}\b", text), name
    assert lib.rk_imt_parser_words() == layout.IP_WORDS and lib.rk_imt_parser_bytes(5) == 5 * 48
    assert lib.rk_adh_state_words() == layout.HS_WORDS and lib.rk_adh_state_bytes(3) == 3 * 48
    assert lib.rk_rmt_state_words() == layout.RS_WORDS and lib.rk_rmt_state_bytes(7) == 7 * 16
    p = _cabi.RmtParams()
    lib.rk_rmt_default_params(C.byref(p))
    assert (p.no_cmd_stop_thre, p.wall_leave_time_ms, p.wall_leave_speed_mmps) == (200, 200, 100)  # RM_task_main.cpp:62-64
    import torch

    if not torch.cuda.is_available():  # no CPU fallback on the new entry points either
        buf = (C.c_uint32 * 256)()
        addr = (C.addressof(buf) + 15) & ~15
        a = C.c_void_p(addr)
        assert lib.rk_rmt_guard(C.byref(p), a, 1, 1, a, a, None, None) == 2
        assert lib.rk_imt_feed_bytes(a, a, 1, 1, 1, a, None, None, None, 0, None) == 2
        assert lib.rk_adh_mode_init(a, 1, 1, None) == 2
        h = C.c_void_p()
        assert lib.rk_rmt_create(C.byref(h), None) == 2


def test_no_cpu_fallback(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    rc = lib.rk_vdt_create(C.byref(h), None)
    assert rc == 2  # RK_ERR_CUDA
    assert b"no CPU fallback" in lib.rk_last_error()
    a = _cabi.VdtRollout()
    a.steps = 1
    buf = (C.c_uint32 * 448)()
    addr = (C.addressof(buf) + 15) & ~15
    rc = lib.rk_vdt_rollout(C.byref(rk.default_params()), C.c_void_p(addr), 1, C.byref(a), None)
    assert rc == 2


def test_argument_errors(lib):
    a = _cabi.VdtRollout()
    a.steps = 1
    rc = lib.rk_vdt_rollout(C.byref(rk.default_params()), C.c_void_p(8), 1, C.byref(a), None)
    assert rc == 1 and b"16-byte aligned" in lib.rk_last_error()
    rc = lib.rk_vdt_rollout(C.byref(rk.default_params()), None, -1, C.byref(a), None)
    assert rc == 1
    # empty batch / zero steps are no-ops
    assert lib.rk_vdt_rollout(C.byref(rk.default_params()), None, 0, C.byref(a), None) == 0


def test_ctypes_structs_match_the_header(tmp_path):
    """Every structure that crosses the C-ABI has the same size and field offsets in _cabi.py as in include/robotick.h
    (compiled with gcc): a field missing on the Python side would silently be read as garbage by the library."""
    import ctypes as C
    import subprocess

    structs = {"rk_vdt_params_t": _cabi.VdtParams, "rk_vdt_rollout_t": _cabi.VdtRollout, "rk_adt_params_t": _cabi.AdtParams,
               "rk_tick_rollout_t": _cabi.TickRollout, "rk_stream_desc_t": _cabi.StreamDesc, "rk_adt_poscmdseq_t": _cabi.AdtPosCmdSeq,
               "rk_rmt_params_t": _cabi.RmtParams, "rk_vdt_cmd_t": _cabi.VdtCmd}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "robotick.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    seen = 0
    for line in out.splitlines():
        cname, fname, val = line.split()
        cls = structs[cname]
        if fname == "size":
            assert C.sizeof(cls) == int(val), f"sizeof({cname}): header {val}, ctypes {C.sizeof(cls)}"
        else:
            assert getattr(cls, fname).offset == int(val), f"{cname}.{fname}: header {val}, ctypes {getattr(cls, fname).offset}"
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in structs.values())


def test_float_encoder_step_is_exact():
    """The packed vehicle tick forms the plant's encoder step rpm * 8192 / 60000 (C truncating division) in float as
    trunc(RN(rpm * C)), C = RN(8192 / 60000) (the float encoder step in fast_tick2, rk_vehicle_fast2.cuh): equal for every
    int16 rpm.  The same check runs on the device before the fast path is enabled (rk_exact.cu)."""
    rw = np.arange(-32768, 32768, dtype=np.int64)
    want = np.sign(rw) * ((np.abs(rw) * 8192) // 60000)
    c = np.float32(0.13653333485126495)
    assert c == np.float32(8192 / 60000)
    got = np.trunc((rw.astype(np.float32) * c).astype(np.float32)).astype(np.int64)
    np.testing.assert_array_equal(got, want)
