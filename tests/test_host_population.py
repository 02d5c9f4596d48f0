"""Host-side checks of the population C ABI and of ``PPOPopulation``'s argument checks (no GPU needed)."""

from __future__ import annotations

import ctypes

import pytest

from rl_brain_trainer_b200 import _lib


def test_member_descriptor_layout_and_entry_points():
    M = _lib.c_struct("KinPopMember")
    H = _lib.c_struct("KinPpoHyper")
    assert _lib.define("KIN_POP_MAX") == 64
    assert M.hyper.offset % 8 == 0 and ctypes.sizeof(M) == M.hyper.offset + ctypes.sizeof(H) and ctypes.sizeof(M) % 8 == 0
    assert M.noise_seed.size == 8 and M.first_step.size == 4 and M.sampler.offset == 0
    L = _lib.lib()
    for name in ("kin_pop_collect", "kin_pop_bootstrap_list", "kin_pop_gae", "kin_pop_adv_stats", "kin_pop_grad_tc", "kin_pop_adam",
                 "kin_params_device_sampler", "kin_params_same_env"):
        assert name in _lib.declared_functions() and hasattr(L, name)


def test_population_launches_reject_bad_arguments_before_touching_the_device():
    L = _lib.lib()
    fake = ctypes.c_void_p(4096)
    hypers = (_lib.c_struct("KinPpoHyper") * 2)()
    steps = (ctypes.c_int * 2)(1, 0)
    cases = [
        lambda: L.kin_pop_collect(None, fake, 1, 256, 0, 16, None),                 # no env handle
        lambda: L.kin_pop_bootstrap_list(fake, 0, 128, None),                       # no members
        lambda: L.kin_pop_gae(fake, 65, 256, 16, None),                             # more than KIN_POP_MAX
        lambda: L.kin_pop_gae(fake, 1, 100, 1, None),                               # tile sums need multiples of 64 samples
        lambda: L.kin_pop_adv_stats(None, 1, 8, 4, None),
        lambda: L.kin_pop_grad_tc(fake, 1, 0, 7, 448, 148, None),                   # odd tile count
        lambda: L.kin_pop_grad_tc(fake, 1, -1, 8, 512, 148, None),
        lambda: L.kin_pop_adam(fake, 2, hypers, steps, None),                       # step 0
        lambda: L.kin_params_device_sampler(None, ctypes.byref(ctypes.c_void_p())),
        lambda: L.kin_params_same_env(None, None, ctypes.byref(ctypes.c_int())),
    ]
    for i, call in enumerate(cases):
        assert call() == _lib.define("KIN_ERR_INVALID_ARG"), i


def test_params_same_env_compares_the_env_params():
    from rl_brain_trainer_b200 import config as kcfg
    from rl_brain_trainer_b200 import params as kparams

    L = _lib.lib()
    handles = []
    for preset in ("approach_default", "approach_default", "approach_dynamic_scale_big"):
        p = kparams.env_params(kcfg.load_preset(preset))
        h = ctypes.c_void_p()
        _lib.check(L.kin_params_create(ctypes.byref(p), ctypes.byref(h)))
        handles.append(h)
    try:
        same = ctypes.c_int(-1)
        _lib.check(L.kin_params_same_env(handles[0], handles[1], ctypes.byref(same)))
        assert same.value == 1
        _lib.check(L.kin_params_same_env(handles[0], handles[2], ctypes.byref(same)))
        assert same.value == 0
        sp = ctypes.c_void_p(1)
        _lib.check(L.kin_params_device_sampler(handles[0], ctypes.byref(sp)))
        assert sp.value is None          # no sampler uploaded yet
    finally:
        for h in handles:
            L.kin_params_destroy(h)


def test_population_needs_trainers():
    from rl_brain_trainer_b200.population import PPOPopulation

    with pytest.raises(ValueError, match="at least one"):
        PPOPopulation([])
    with pytest.raises(TypeError, match="PPOTrainer"):
        PPOPopulation([object()])
    with pytest.raises(ValueError, match="KIN_POP_MAX"):
        PPOPopulation([object()] * 65)
