"""Every C entry point that takes an rt_ray_desc checks the batch and resolves its window the same way: the return
code of each malformed descriptor or window, and which checks come before the NULL-pointer checks and device work.
Called with host buffers on a machine without a device, so a call that passes every check ends in RT_ERR_CUDA (-2)."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="a well-formed call would launch on host pointers")

INF = float("inf")


@pytest.fixture(scope="module")
def lib():
    from triro.backend import build, ops

    build.build()
    return ops.get_module()


@pytest.fixture(scope="module")
def addr():
    buf = (C.c_uint8 * 8192)()
    return (C.addressof(buf) + 255) // 256 * 256, buf          # 256-byte aligned (scene tables), kept alive


def _f3():
    return (C.c_float * 3)(1.0, 0.0, 0.0)


# name -> (column of the expected-code table, call(lib, a, rd, opts)); a is an aligned host address for every buffer
ENTRY = {
    "rt_trace_any": ("trace", lambda L, a, rd, o: L.rt_trace_any(a, rd, o, a, a, None)),
    "rt_trace_first": ("trace", lambda L, a, rd, o: L.rt_trace_first(a, rd, o, a, a, None)),
    "rt_trace_closest": ("trace", lambda L, a, rd, o: L.rt_trace_closest(a, rd, o, a, a, a, a, a, a, None)),
    "rt_trace_count": ("trace", lambda L, a, rd, o: L.rt_trace_count(a, rd, o, a, a, None)),
    "rt_contains_parity": ("clears", lambda L, a, rd, o: L.rt_contains_parity(a, rd, o, _f3(), _f3(), _f3(), None, a, a, a,
                                                                               a, None)),
    "rt_trace_stats": ("clears", lambda L, a, rd, o: L.rt_trace_stats(a, rd, o, 0, a, a, None)),
    "rt_allhits_trace": ("allhits", lambda L, a, rd, o: L.rt_allhits_trace(a, rd, o, 8, a, a, a, 4096, a, a, None)),
    "rt_closest_point": ("point", lambda L, a, rd, o: L.rt_closest_point(a, rd, o, INF, a, a, a, a, None, a, None)),
    "rt_signed_distance": ("point", lambda L, a, rd, o: L.rt_signed_distance(a, a, rd, o, a, None, a, None)),
    "rt_signed_distance_closest": ("point", lambda L, a, rd, o: L.rt_signed_distance_closest(a, a, rd, o, a, a, a, a, None,
                                                                                               a, None)),
    "rt_winding_number": ("point", lambda L, a, rd, o: L.rt_winding_number(a, a, rd, o, 2.0, a, None, a, None)),
    "rt_scene_trace": ("point", lambda L, a, rd, o: L.rt_scene_trace(a, a, rd, o, 0, a, a, a, a, a, a, a, None)),
    "rt_scene_closest_point": ("point", lambda L, a, rd, o: L.rt_scene_closest_point(a, a, a, rd, o, INF, a, a, a, a, a,
                                                                                       None)),
    "rt_scene_signed_distance": ("point", lambda L, a, rd, o: L.rt_scene_signed_distance(a, a, a, a, rd, o, a, None, None,
                                                                                           None, None, None)),
    # grad_points only: one launch, no workspace
    "rt_distance_grad": ("point", lambda L, a, rd, o: L.rt_distance_grad(rd, o, a, a, a, a, a, a, 1, 3, a, None, None, 0,
                                                                         None)),
    # one hit row, no row_ray: the rows must be the window's rays
    "rt_ray_grad": ("raygrad", lambda L, a, rd, o: L.rt_ray_grad(rd, o, 1, None, a, a, a, a, 3, a, 1, a, a, None, None, 0,
                                                                 None)),
    # one instance of one 3-vertex member; grad_origins only, no workspace
    "rt_scene_ray_grad": ("raygrad", lambda L, a, rd, o: L.rt_scene_ray_grad(a, 1, a, 1, 3, rd, o, 1, None, a, a, a, a, a,
                                                                             None, None, None, None, 0, None)),
    # grad_points only, no workspace
    "rt_scene_distance_grad": ("point", lambda L, a, rd, o: L.rt_scene_distance_grad(a, 1, a, 1, 3, rd, o, a, a, a, a, a,
                                                                                       a, a, None, None, None, 0, None)),
}

# case -> (descriptor edit, (ray_first, ray_count) or None for NULL opts, expected code per column)
CASES = {
    "whole_batch": ({}, None, dict(trace=-2, allhits=-2, point=-2, raygrad=-2)),
    "empty_window": ({}, (1, -1), dict(trace=0, allhits=-2, point=0, raygrad=-1)),
    "ray_first_past_end": ({}, (2, -1), dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
    "window_past_end": ({}, (0, 2), dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
    "nray_not_shape": ({"nray": 2}, None, dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
    "last_dim_4": ({"shape3": 4}, None, dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
    "negative_nray": ({"nray": -1}, None, dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
    "null_origins": ({"origins": None}, None, dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
    "null_origins_empty_window": ({"origins": None}, (1, -1), dict(trace=-1, allhits=-1, point=0, raygrad=-1)),
    "null_descriptor": (None, None, dict(trace=-1, allhits=-1, point=-1, raygrad=-1)),
}


def _desc(a, edit):
    from triro.backend import ops

    rd = ops.RayDesc()
    rd.nray = edit.get("nray", 1)
    for i, s in enumerate((1, 1, 1, edit.get("shape3", 3))):
        rd.shape[i] = s
    rd.o_stride[3] = rd.d_stride[3] = 1
    rd.origins = edit.get("origins", a)
    rd.directions = a
    return rd


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("name", list(ENTRY))
def test_batch_and_window_checks(lib, addr, name, case):
    from triro.backend import ops

    a = addr[0]
    column, call = ENTRY[name]
    edit, window, expect = CASES[case]
    rd = None if edit is None else C.byref(_desc(a, edit))
    opts = None if window is None else C.byref(ops.trace_opts(None, *window))
    # rt_contains_parity and rt_trace_stats clear a device buffer before any check
    want = -2 if column == "clears" else expect[column]
    rc = call(lib, a, rd, opts)
    msg = lib.rt_last_error()
    assert rc == want, (rc, msg)
    if rc == -1:
        assert msg.startswith(name.encode() + b":"), msg
        if case == "ray_first_past_end":
            assert b"ray_first" in msg, msg
