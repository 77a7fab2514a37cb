"""CPU tests of the mixed scene (vfk_buffers.obst_shared = 2): the appended ABI fields and the workload builders."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
APPENDED = ("shared_obst", "shared_obst_ext", "n_shared_obst", "reserved2")


def test_appended_buffer_fields_match_the_header(tmp_path):
    """offsetof of every mixed-scene field of vfk_buffers, from a C compiler reading include/vfk.h, against BuffersC; the
    fields sit after every older one, and the mode constants agree."""
    from vfclik_b200 import _lib
    prog = tmp_path / "offsets.c"
    fields = ("jp_hi",) + APPENDED
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vfk.h"\n'
                    'int main(void){printf("%zu' + ' %zu' * len(fields) + ' %d %d %d\\n", sizeof(vfk_buffers), '
                    + ", ".join("offsetof(vfk_buffers, %s)" % f for f in fields)
                    + ', VFK_OBST_PER_INSTANCE, VFK_OBST_SHARED, VFK_OBST_MIXED); return 0;}\n')
    exe = tmp_path / "offsets"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got[0] == C.sizeof(_lib.BuffersC)
    assert got[1:1 + len(fields)] == [getattr(_lib.BuffersC, f).offset for f in fields]
    assert got[2] > got[1]                       # appended after the last field of the older struct
    assert got[1 + len(fields):] == [_lib.VFK_OBST_PER_INSTANCE, _lib.VFK_OBST_SHARED, _lib.VFK_OBST_MIXED] == [0, 1, 2]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("ext", [False, True])
def test_mixed_scene_batch_and_concat(dtype, ext):
    from vfclik_b200 import workloads
    chain = workloads.dual_arm_torso_chain(7)
    n, Mi, Ms = 70, 5, 3
    w = workloads.mixed_scene_batch(chain, n, Mi, Ms, seed=4, dtype=dtype, obst_ext=ext)
    assert w["q"].shape == (7, n) and w["goal"].shape == (13, n)
    assert w["obst"].shape == (Mi, n, 4) and w["shared_obst"].shape == (Ms, 4)
    assert all(v.dtype == dtype for v in w.values())
    assert ("obst_ext" in w) == ext and ("shared_obst_ext" in w) == ext
    if ext:
        assert w["obst_ext"].shape == (Mi, n, 2) and w["shared_obst_ext"].shape == (Ms, 2)
    # starts, goals and own obstacles are random_batch's with the seed; the shared list is its single-instance draw
    ref = workloads.random_batch(chain, n, Mi, 4, dtype=dtype, obst_ext=ext)
    assert np.array_equal(w["q"], ref["q"]) and np.array_equal(w["obst"], ref["obst"])
    one = workloads.random_batch(chain, 1, Ms, 5, dtype=dtype)
    assert np.array_equal(w["shared_obst"], one["obst"][:, 0])
    c = workloads.concat_scene(w["obst"], w["shared_obst"], n)
    assert c.shape == (Mi + Ms, n, 4) and c.dtype == dtype and c.flags.c_contiguous
    assert np.array_equal(c[:Mi], w["obst"])
    assert np.array_equal(c[Mi:], np.broadcast_to(w["shared_obst"][:, None], (Ms, n, 4)))
    if ext:
        ce = workloads.concat_scene(w["obst_ext"], w["shared_obst_ext"], n)
        assert ce.shape == (Mi + Ms, n, 2) and np.array_equal(ce[Mi:, 7], w["shared_obst_ext"])
    # degenerate lists
    assert workloads.concat_scene(np.zeros((0, n, 4), dtype), w["shared_obst"], n).shape == (Ms, n, 4)
    assert workloads.concat_scene(w["obst"], np.zeros((0, 4), dtype), n).shape == (Mi, n, 4)
    with pytest.raises(ValueError):
        workloads.concat_scene(w["obst"], w["shared_obst"], n + 1)
