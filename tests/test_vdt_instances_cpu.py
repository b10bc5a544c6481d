"""CPU: every vehicle rollout instantiation compiled into the library is one the GPU matrix of test_vdt_instances_gpu.py
launches (so a new instantiation cannot ship untested), and rk_set_option's host-side validation."""
import pytest

import vdt_instances as vi
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi

RK_ERR_ARG = 1


def test_parse_accepts_both_demangler_spellings():
    cu = "void rk::vdt_rollout_fast_kernel<(bool)0, (int)3, (int)2, (bool)1, (bool)0, (bool)1, (int)2>(rk_vdt_params, uint4 *, long)"
    cxx = "void rk::vdt_rollout_fast_kernel<false, 3, 2, true, false, true, 2>(rk_vdt_params_t, uint4*, long)"
    mangled = "_ZN2rk23vdt_rollout_fast_kernelILb0ELi3ELi2ELb1ELb0ELb1ELi2EEEv13rk_vdt_paramsP5uint4l"
    assert vi.parse(cu) == vi.parse(cxx) == vi.parse(mangled) == ("fast", 0, 3, 2, 1, 0, 1, 2)
    assert vi.parse("void rk::vdt_rollout_stream_fast_kernel<true, 3>(rk_vdt_params)") == ("stream", 1, 3)
    assert vi.parse("void rk::vdt_rollout_kernel<(int)2, (bool)1, (bool)0, (int)0>(rk_vdt_params)") == ("transcription", 2, 1, 0, 0)
    assert vi.parse("void rk::vdt_set_power_kernel(uint4 *, long, const unsigned char *)") is None


def test_expected_kernel_restates_the_dispatch():
    e = vi.expected_kernel
    assert e("plant") == ("fast", 0, 4, 2, 1, 0, 0, 0)
    assert e("plant", reset_state=True) == ("fast", 0, 4, 2, 1, 1, 0, 0)  # the one reset-in-kernel instantiation
    assert e("plant", reset_state=True, occupancy=3) == ("fast", 0, 3, 2, 1, 0, 0, 0)
    assert e("plant", reset_state=True, kd=0.0005) == ("fast", 0, 4, 0, 1, 0, 0, 0)
    assert e("plant", reset_state=True, trace=True) == ("fast", 1, 4, 2, 1, 0, 0, 0)
    assert e("plant", trace=True, occupancy=3, ffsat=1) == ("fast", 1, 4, 3, 1, 0, 0, 0)  # traced: occupancy 4 only
    assert e("plant", packed=0, ffsat=1) == ("fast", 0, 4, 1, 0, 0, 0, 0)  # scalar: no KD0
    assert e("plant", ffsat=1, ff_limit=0.5) == ("fast", 0, 4, 2, 1, 0, 0, 0)  # FFSAT needs ff_limit == 1
    assert e("stream", packed=0, occupancy=3, ffsat=1) == ("stream", 0, 3)
    assert e("moving", occupancy=3, packed=0, kd=0.0005) == ("fast", 0, 3, 0, 0, 0, 1, 2)
    assert e("obstacles", force_transcription=1) == ("transcription", 1, 0, 1, 1)
    assert e("plant", fast_usable=False, trace=True) == ("transcription", 1, 1, 0, 0)
    assert e("hold", trace=True) == ("transcription", 0, 1, 0, 0)


def test_every_compiled_instantiation_is_launched_by_the_matrix():
    if vi.tool("cuobjdump") is None or vi.tool("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not found")
    rk.load()  # the library is built
    compiled = vi.inventory()
    declared = vi.declared()
    assert len(compiled) == 72, f"{len(compiled)} vehicle rollout instantiations compiled: {sorted(compiled)}"
    untested = sorted(compiled - set(declared))
    assert not untested, f"compiled but launched by no row of the matrix: {untested}"
    missing = sorted((k, declared[k]) for k in set(declared) - compiled)
    assert not missing, f"the matrix expects instantiations the library does not contain: {missing}"


@pytest.fixture
def lib():
    lib = rk.load()
    yield lib
    for opt, v in ((_cabi.RK_OPT_FAST_OCCUPANCY, 4), (_cabi.RK_OPT_STREAM_CTAS, 0), (_cabi.RK_OPT_TICK_SIDE_CTAS, 0)):
        assert lib.rk_set_option(opt, v) == _cabi.RK_OK


def test_set_option_ranges(lib):
    ok, bad = _cabi.RK_OK, RK_ERR_ARG
    cases = [(_cabi.RK_OPT_FAST_OCCUPANCY, v, ok) for v in (3, 4)]
    cases += [(_cabi.RK_OPT_FAST_OCCUPANCY, v, bad) for v in (2, 5, 0, -4)]
    cases += [(_cabi.RK_OPT_STREAM_CTAS, v, ok) for v in (0, 1, 32, -1, -100000)]  # < 0: -v CTAs in all
    cases += [(_cabi.RK_OPT_STREAM_CTAS, v, bad) for v in (33, -100001)]
    cases += [(_cabi.RK_OPT_TICK_SIDE_CTAS, v, ok) for v in (0, 1, 8)]
    cases += [(_cabi.RK_OPT_TICK_SIDE_CTAS, v, bad) for v in (-1, 9)]
    cases += [(0, 1, bad), (7, 0, bad), (-1, 0, bad)]  # unknown options
    got = [(opt, v, lib.rk_set_option(opt, v)) for opt, v, _ in cases]
    assert got == cases
