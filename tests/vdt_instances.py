"""TEST INFRASTRUCTURE: the vehicle rollout's compiled kernel instantiations and the dispatch that picks one.

rk_vdt_rollout and rk_plan_rollout* choose a template instantiation of one of three kernels from the params and the
process-wide RK_OPT_* options (fast_cfg, with_fast_cfg, launch_plan and the reset_in_kernel rule in rk_vehicle.cu):

    ("fast", TRACE, OCC, FLAGS, PACKED, RESET, PLAN, OBST)   vdt_rollout_fast_kernel
    ("stream", TRACE, FLAGS)                                 vdt_rollout_stream_fast_kernel
    ("transcription", MODE, TRACE, PLAN, OBST)               vdt_rollout_kernel

FLAGS bit 0 is FFSAT (the FMUL.SAT form of the feed-forward clamp), bit 1 KD0 (kd == 0).  inventory() lists what the
built library contains; expected_kernel() restates the dispatch, so that a test can assert which instantiation ran.
Shared by test_vdt_instances_cpu.py and test_vdt_instances_gpu.py.
"""
import os
import re
import shutil
import subprocess

from roboken_fmskf_robot_controller_b200 import _cabi

KINDS = {"vdt_rollout_fast_kernel": "fast", "vdt_rollout_stream_fast_kernel": "stream", "vdt_rollout_kernel": "transcription"}
_DEMANGLED = re.compile(r"rk::(vdt_rollout(?:_stream)?(?:_fast)?_kernel)<([^>]*)>")
_MANGLED = re.compile(r"_ZN2rk\d+(vdt_rollout(?:_stream)?(?:_fast)?_kernel)I((?:L[bi]\d+E)+)E")
_ARG = {"true": 1, "false": 0}

ENTRY_OBST = {"plan": 0, "obstacles": 1, "moving": 2}  # rk_plan_rollout, _obstacles, _moving (with m > 0 or a path)
MODES = {"hold": _cabi.RK_SENSOR_HOLD, "plant": _cabi.RK_SENSOR_PLANT, "stream": _cabi.RK_SENSOR_STREAM}


def _arg(s):
    """One template argument as either demangler spells it: (bool)1, true, (int)3, 3."""
    s = re.sub(r"^\((?:bool|int)\)", "", s.strip())
    return _ARG[s] if s in _ARG else int(s)


def parse(name):
    """A kernel name (demangled by cu++filt or c++filt, or mangled) -> its instantiation tuple, or None for any other
    kernel."""
    m = _DEMANGLED.search(name)
    if m:
        return (KINDS[m.group(1)],) + tuple(_arg(a) for a in m.group(2).split(","))
    m = _MANGLED.search(name)
    if m:
        return (KINDS[m.group(1)],) + tuple(int(v) for v in re.findall(r"L[bi](\d+)E", m.group(2)))
    return None


def toolkit_bin():
    """The directory of the toolkit that builds the library: $NVCC's, else /usr/local/cuda/bin."""
    nvcc = os.environ.get("NVCC")
    return os.path.dirname(nvcc) if nvcc else "/usr/local/cuda/bin"


def tool(name):
    path = os.path.join(toolkit_bin(), name)
    return path if os.path.exists(path) else shutil.which(name)


def inventory(lib_path=_cabi.LIB_PATH):
    """The set of vehicle rollout instantiations compiled into the library (cuobjdump -symbols | cu++filt)."""
    dump = subprocess.run([tool("cuobjdump"), "-symbols", lib_path], check=True, capture_output=True, text=True).stdout
    names = subprocess.run([tool("cu++filt")], input=dump, check=True, capture_output=True, text=True).stdout
    return {t for t in map(parse, names.splitlines()) if t is not None}


def expected_kernel(entry, *, occupancy=4, packed=1, ffsat=0, force_transcription=0, kd=0.0, ff_limit=1.0, fast_usable=True,
                    trace=False, reset_state=False):
    """The instantiation rk_vdt_rollout (entry "hold", "plant" or "stream") or rk_plan_rollout* (entry "plan",
    "obstacles" or "moving") launches.  Options: RK_OPT_FAST_OCCUPANCY, _FAST_PACKED, _FAST_FFSAT, _FORCE_TRANSCRIPTION.
    Params: kd, ff_limit, and fast_usable = whether the params pass the fast path's host checks and on-device proofs."""
    plan = entry in ENTRY_OBST
    obst = ENTRY_OBST.get(entry, 0)
    mode = _cabi.RK_SENSOR_PLANT if plan else MODES[entry]
    if plan:
        trace, reset_state = False, False
    fast = fast_usable and not force_transcription and mode != _cabi.RK_SENSOR_HOLD
    if not fast:
        return ("transcription", mode, int(trace), int(plan), obst)
    stream = mode == _cabi.RK_SENSOR_STREAM
    occ = 4 if (trace or occupancy != 3) else 3  # traced kernels are compiled at occupancy 4 only
    pk = 1 if (stream or packed) else 0  # the stream kernel has no scalar form
    flags = (1 if (ff_limit == 1.0 and ffsat) else 0) | (2 if (kd == 0.0 and pk) else 0)  # KD0: packed tick only
    if stream:
        return ("stream", int(trace), flags)
    # only the default packed untraced configuration has a kernel that starts from zeros in registers; every other
    # reset_state launch is a memset and then the ordinary kernel
    reset_in_kernel = reset_state and not plan and not trace and occ == 4 and flags == 2 and pk
    return ("fast", int(trace), occ, flags, pk, int(reset_in_kernel), int(plan), obst)


# ---- the matrix test_vdt_instances_gpu.py runs ------------------------------------------------------------------------
# One row: the options and params of one case.  kd = 0.0005 turns KD0 off; ff_limit = 0.5 keeps FFSAT from applying even
# with RK_OPT_FAST_FFSAT on.
PARAMS = [dict(kd=kd, ff_limit=ff) for kd in (0.0, 0.0005) for ff in (1.0, 0.5)]
MATRIX = [dict(occupancy=occ, packed=pk, ffsat=fs, force_transcription=0, **pr)
          for occ in (3, 4) for pk in (0, 1) for fs in (0, 1) for pr in PARAMS]
MATRIX += [dict(occupancy=4, packed=1, ffsat=0, force_transcription=1, **pr) for pr in PARAMS]
# The launches each row's battery makes, as (entry, trace, reset_state); the GPU test checks that it makes exactly these.
BATTERY = {("hold", True, False), ("hold", False, False),
           ("plant", True, False), ("plant", False, False), ("plant", True, True), ("plant", False, True),
           ("stream", True, False), ("stream", False, False),
           ("plan", False, False), ("obstacles", False, False), ("moving", False, False)}


def row_id(row):
    if row["force_transcription"]:
        return f"transcription-kd{row['kd']:g}-ff{row['ff_limit']:g}"
    return f"occ{row['occupancy']}-{'packed' if row['packed'] else 'scalar'}-ffsat{row['ffsat']}-kd{row['kd']:g}-ff{row['ff_limit']:g}"


def declared():
    """Every instantiation the matrix launches, with the first row that launches it."""
    out = {}
    for row in MATRIX:
        for entry, trace, reset in sorted(BATTERY):
            out.setdefault(expected_kernel(entry, trace=trace, reset_state=reset, **row), row_id(row))
    return out
