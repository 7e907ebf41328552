"""Actuator latency and joint-angle observation noise without a GPU: Sim2Real parsing and validation, the ctypes mirrors of
so100_sim2real / so100_actuator_view against the header, and argument checks of the new entry points."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from so100_mujoco_rl_b200.randomization import ACTUATOR_NAMES, Sim2Real, So100ActuatorView, So100Sim2Real


def test_defaults_are_off_and_scalars_broadcast():
    s = Sim2Real()
    assert s.latency == (0, 0)
    np.testing.assert_array_equal(s.obs_noise, np.zeros(6))
    s = Sim2Real(latency=(2, 9), obs_noise=0.01)
    assert s.latency == (2, 9)
    np.testing.assert_array_equal(s.obs_noise, [0.01] * 6)
    per = [0.0, 0.01, 0.02, 0.0, 0.005, 0.1]
    np.testing.assert_array_equal(Sim2Real(obs_noise=per).obs_noise, per)


@pytest.mark.parametrize("lat", [(-1, 0), (3, 2), (0.5, 2), (0, 2.0), (1,), (0, 1, 2), (True, 2)])
def test_bad_latency_is_rejected(lat):
    with pytest.raises(ValueError):
        Sim2Real(latency=lat)


def test_latency_bounds_follow_the_model():
    Sim2Real(latency=(0, 16)).validate()  # the so100 model: 16 substeps
    Sim2Real(latency=(16, 16)).validate(nsubstep=16)
    Sim2Real(latency=(0, 20)).validate(nsubstep=20)
    for lat in ((0, 17), (17, 17)):
        with pytest.raises(ValueError):
            Sim2Real(latency=lat).validate()
    with pytest.raises(ValueError):
        Sim2Real(latency=(0, 9)).validate(nsubstep=8)


@pytest.mark.parametrize("noise", [-0.01, float("nan"), float("inf"), 1e39, [0.01] * 5, [[0.01] * 6],
                                   [0.0, 0.0, -1e-9, 0.0, 0.0, 0.0]])
def test_bad_noise_is_rejected(noise):
    with pytest.raises(ValueError):
        Sim2Real(obs_noise=noise)


def test_env05_takes_latency_but_no_noise():
    Sim2Real(latency=(0, 16)).validate(task=5)
    Sim2Real(latency=(0, 16), obs_noise=0.0).validate(task=5)
    for t in (1, 2, 6):
        Sim2Real(obs_noise=0.02).validate(task=t)
    with pytest.raises(ValueError):
        Sim2Real(obs_noise=0.02).validate(task=5)
    with pytest.raises(ValueError):
        Sim2Real(obs_noise=[0, 0, 0, 0, 0, 1e-3]).validate(task=5)


def test_parse_latency():
    assert Sim2Real.parse_latency("0:8") == (0, 8)
    assert Sim2Real.parse_latency(" 3 ") == (3, 3)
    for bad in ("a:b", "1.5:2", "", "1:"):
        with pytest.raises(ValueError):
            Sim2Real.parse_latency(bad)


def test_to_ctypes_and_dict_roundtrip():
    s = Sim2Real(latency=(1, 7), obs_noise=[0.0, 0.01, 0.02, 0.03, 0.04, 0.05])
    c = s.to_ctypes()
    assert c.struct_size == ctypes.sizeof(So100Sim2Real) == 16 + 6 * 8
    assert tuple(c.latency) == (1, 7) and c.obs_noise[0] == 0.0 and c.obs_noise[5] == 0.05
    d = s.to_dict()
    assert d == {"latency": [1, 7], "obs_noise": [0.0, 0.01, 0.02, 0.03, 0.04, 0.05]}
    back = Sim2Real.from_dict(d)
    assert back.latency == s.latency and (back.obs_noise == s.obs_noise).all()


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
  printf("%zu %zu %zu %zu %zu\\n", sizeof(so100_sim2real), offsetof(so100_sim2real, struct_size), offsetof(so100_sim2real, latency),
         offsetof(so100_sim2real, _pad0), offsetof(so100_sim2real, obs_noise));
  printf("%zu %zu %zu %zu\\n", sizeof(so100_actuator_view), offsetof(so100_actuator_view, latency),
         offsetof(so100_actuator_view, ctrl_prev_hi), offsetof(so100_actuator_view, ctrl_prev_lo));
  return 0;
}
""")
    exe = tmp_path / "layout"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    a, b = subprocess.check_output([str(exe)], text=True).splitlines()
    want_a = [ctypes.sizeof(So100Sim2Real)] + [getattr(So100Sim2Real, f).offset for f in ("struct_size", "latency", "_pad0", "obs_noise")]
    want_b = [ctypes.sizeof(So100ActuatorView)] + [getattr(So100ActuatorView, f).offset for f in ACTUATOR_NAMES]
    assert [int(x) for x in a.split()] == want_a
    assert [int(x) for x in b.split()] == want_b


def test_new_entry_points_reject_null_arguments(native_lib):
    s = Sim2Real(latency=(0, 4)).to_ctypes()
    v = So100ActuatorView()
    assert native_lib.so100_set_sim2real(None, ctypes.byref(s)) == -1
    assert native_lib.so100_set_sim2real(None, None) == -1
    assert native_lib.so100_get_actuator_state(None, ctypes.byref(v), None) == -1
    assert native_lib.so100_set_actuator_state(None, ctypes.byref(v), None) == -1
    assert native_lib.so100_get_actuator_state(None, None, None) == -1
    assert native_lib.so100_set_actuator_state(None, None, None) == -1
    assert b"null argument" in native_lib.so100_last_error()
