"""Host-side checks of the route-population C ABI (``KinPopRouteMember`` and the ``kin_pop_route_*`` entry points) and of
``PPOPopulation.build``'s route arguments (no GPU needed)."""

from __future__ import annotations

import ctypes

import pytest

from rl_brain_trainer_b200 import _lib


def test_route_member_descriptor_layout_and_entry_points():
    R = _lib.c_struct("KinPopRouteMember")
    C = _lib.c_struct("KinRouteResetParams")
    assert R.obs.offset == 0 and R.route_flags.offset == 8 and R.reset.offset == 16
    assert ctypes.sizeof(C) == 84 and ctypes.sizeof(R) == 16 + 84 + 4 and ctypes.sizeof(R) % 8 == 0
    assert ctypes.sizeof(_lib.c_struct("KinPopMember")) == 296         # the arm descriptor keeps its layout
    assert _lib.define("KIN_ABI_VERSION") == 4
    L = _lib.lib()
    for name in ("kin_pop_route_collect", "kin_pop_route_bootstrap_list", "kin_pop_route_obs_images", "kin_pop_route_logp",
                 "kin_pop_route_grad_tc", "kin_pop_route_adam"):
        assert name in _lib.declared_functions() and hasattr(L, name)


def test_route_population_launches_reject_bad_arguments_before_touching_the_device():
    L = _lib.lib()
    fake = ctypes.c_void_p(4096)           # never dereferenced: every call below fails its argument checks first
    hypers = (_lib.c_struct("KinPpoHyper") * 2)()
    steps = (ctypes.c_int * 2)(1, 0)
    table = _lib.c_struct("KinRouteTable")()
    cases = [
        lambda: L.kin_pop_route_collect(None, ctypes.byref(table), fake, fake, 1, 256, 16, 0, 1, 1, None),    # no env handle
        lambda: L.kin_pop_route_collect(None, None, fake, fake, 1, 256, 16, 0, 1, 1, None),                   # no route table
        lambda: L.kin_pop_route_bootstrap_list(None, 1, 256, 128, 0, None),
        lambda: L.kin_pop_route_bootstrap_list(fake, 65, 256, 128, 0, None),                                  # more than KIN_POP_MAX
        lambda: L.kin_pop_route_bootstrap_list(fake, 1, 256, 128, -16, None),                                 # negative chunk offset
        lambda: L.kin_pop_route_bootstrap_list(fake, 1, 0, 128, 0, None),
        lambda: L.kin_pop_route_obs_images(fake, None, 1, 4096, None),                                        # no route table
        lambda: L.kin_pop_route_obs_images(fake, fake, 1, 4000, None),                                        # rows not a multiple of 128
        lambda: L.kin_pop_route_logp(fake, 1, None, 64, 148, None),                                           # no tile list
        lambda: L.kin_pop_route_logp(fake, 1, fake, 63, 148, None),                                           # odd tile count
        lambda: L.kin_pop_route_logp(fake, 1, fake, 64, 0, None),
        lambda: L.kin_pop_route_grad_tc(fake, 1, 0, 7, 448, 148, None),                                       # odd tile count
        lambda: L.kin_pop_route_grad_tc(fake, 1, -1, 8, 512, 148, None),
        lambda: L.kin_pop_route_grad_tc(fake, 0, 0, 8, 512, 148, None),
        lambda: L.kin_pop_route_adam(fake, 2, hypers, steps, None),                                           # step 0
        lambda: L.kin_pop_route_adam(fake, 2, None, steps, None),
    ]
    for i, call in enumerate(cases):
        assert call() == _lib.define("KIN_ERR_INVALID_ARG"), i


def test_build_rejects_route_curricula_without_a_route():
    from rl_brain_trainer_b200.population import PPOPopulation

    with pytest.raises(ValueError, match="route_curricula needs route="):
        PPOPopulation.build(None, [None], [None], [0], 256, route_curricula=[None])
    with pytest.raises(ValueError, match="one config"):
        PPOPopulation.build(None, [None, None], [None], [0], 256)
