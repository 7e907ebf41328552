"""Per-env dynamics randomisation without a GPU: ParamRanges parsing, broadcasting and validation, the ctypes mirrors of
so100_param_ranges / so100_param_view against the header, and argument checks of the new entry points."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from so100_mujoco_rl_b200.randomization import FIELDS, ParamRanges, So100ParamRanges, So100ParamView, parse


def test_parse_full_spec():
    r = parse("kp=0.7:1.3,damping=0.8:1.2,forcerange=0.8:1.0,frictionloss=0.5:2")
    np.testing.assert_array_equal(r.kp, [[0.7, 1.3]] * 6)
    np.testing.assert_array_equal(r.damping, [[0.8, 1.2]] * 6)
    np.testing.assert_array_equal(r.forcerange, [[0.8, 1.0]] * 6)
    np.testing.assert_array_equal(r.frictionloss, [[0.5, 2.0]] * 6)


def test_parse_leaves_unnamed_fields_at_unit_scale():
    r = ParamRanges.parse(" kp = 0.5:1.5 ")
    np.testing.assert_array_equal(r.kp, [[0.5, 1.5]] * 6)
    for f in ("damping", "forcerange", "frictionloss"):
        np.testing.assert_array_equal(getattr(r, f), [[1.0, 1.0]] * 6)
    assert ParamRanges.parse("").to_dict() == ParamRanges().to_dict()


@pytest.mark.parametrize("spec", ["kp", "kp=1", "kp=a:b", "mass=1:2", "kp=1:2,kp=1:2", "kp=2:1", "kp=0:1", "forcerange=-1:1",
                                  "damping=-0.1:1", "frictionloss=-1:0", "kp=nan:1", "kp=1:inf", "kp=1:1e39"])
def test_bad_specs_are_rejected(spec):
    with pytest.raises(ValueError):
        parse(spec)


def test_zero_lower_bound_is_allowed_for_damping_and_friction_only():
    ParamRanges(damping=(0.0, 1.0), frictionloss=(0.0, 0.0))
    with pytest.raises(ValueError):
        ParamRanges(kp=(0.0, 1.0))
    with pytest.raises(ValueError):
        ParamRanges(forcerange=(0.0, 1.0))


def test_per_joint_ranges_and_broadcasting():
    per = np.array([[0.5 + 0.1 * j, 1.0 + 0.1 * j] for j in range(6)])
    r = ParamRanges(kp=per, damping=[0.9, 1.1])
    np.testing.assert_array_equal(r.kp, per)
    np.testing.assert_array_equal(r.damping, np.tile([0.9, 1.1], (6, 1)))
    bad = per.copy()
    bad[3] = [1.2, 1.1]
    with pytest.raises(ValueError):
        ParamRanges(kp=bad)
    with pytest.raises(ValueError):
        ParamRanges(kp=np.ones((5, 2)))
    lo, hi = r.lo_hi_f32()
    assert lo.dtype == np.float32 and lo.shape == (24,)
    np.testing.assert_array_equal(lo[:6], per[:, 0].astype(np.float32))
    np.testing.assert_array_equal(hi[6:12], np.float32(1.1))


def test_to_ctypes_and_dict_roundtrip():
    r = parse("kp=0.7:1.3,frictionloss=0.5:2")
    c = r.to_ctypes()
    assert c.struct_size == ctypes.sizeof(So100ParamRanges) == 8 + 4 * 6 * 2 * 8
    assert tuple(c.kp[2]) == (0.7, 1.3) and tuple(c.frictionloss[5]) == (0.5, 2.0) and tuple(c.damping[0]) == (1.0, 1.0)
    assert ParamRanges.from_dict(r.to_dict()).to_dict() == r.to_dict()


def test_ctypes_layout_matches_the_header(tmp_path):
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text("""
#include <stddef.h>
#include <stdio.h>
#include "so100_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(so100_param_ranges), offsetof(so100_param_ranges, kp),
         offsetof(so100_param_ranges, damping), offsetof(so100_param_ranges, forcerange), offsetof(so100_param_ranges, frictionloss),
         sizeof(so100_param_view));
  printf("%zu %zu %zu %zu %zu\\n", offsetof(so100_param_view, kp), offsetof(so100_param_view, kv), offsetof(so100_param_view, force_lo),
         offsetof(so100_param_view, force_hi), offsetof(so100_param_view, frictionloss));
  return 0;
}
""")
    exe = tmp_path / "layout"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    a, b = subprocess.check_output([str(exe)], text=True).splitlines()
    want_a = [ctypes.sizeof(So100ParamRanges)] + [getattr(So100ParamRanges, f).offset for f in FIELDS] + [ctypes.sizeof(So100ParamView)]
    want_b = [getattr(So100ParamView, f).offset for f in ("kp", "kv", "force_lo", "force_hi", "frictionloss")]
    assert [int(x) for x in a.split()] == want_a
    assert [int(x) for x in b.split()] == want_b


def test_new_entry_points_reject_null_arguments(native_lib):
    r = ParamRanges().to_ctypes()
    v = So100ParamView()
    assert native_lib.so100_set_param_ranges(None, ctypes.byref(r)) == -1
    assert native_lib.so100_set_param_ranges(None, None) == -1
    assert native_lib.so100_get_env_params(None, ctypes.byref(v), None) == -1
    assert native_lib.so100_set_env_params(None, ctypes.byref(v), None) == -1
    assert native_lib.so100_get_env_params(None, None, None) == -1
    assert b"null argument" in native_lib.so100_last_error()
