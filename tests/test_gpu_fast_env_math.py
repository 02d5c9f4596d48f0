"""The env arithmetic of kin_core.cuh / kin_tc16.cuh on the device, step by step, against fp64 references -- above all the FAST
flavour (sqrt.approx / rcp.approx, the polynomial atan2, MUFU or polynomial sine / cosine, carried pose-error norms, margins from the
normalised q, the packed fp16 observation) that only the tensor-core rollout runs and whose closed-loop tests only see outcomes.

tests/kin_fast_env_harness.cu calls the library's own device functions; it is compiled with the library's nvcc flags into a temporary
directory (cached by a hash of the harness and the headers) and loaded with ctypes.  References: numpy in fp64 on the fp32 inputs,
and the pinned C oracle (ko.fk_pose6, kor_reset, ko.step_batch, kor_observation) with the tolerances of test_gpu_env_parity.py.
"""

from __future__ import annotations

import ctypes
import functools
import hashlib
import os
import subprocess
import tempfile
from dataclasses import replace
from pathlib import Path

import numpy as np
import pytest

from oracle import kin_oracle as ko

from ._util import GOLD, _geodesic, _near, _thresholds, env_config, env_config_from_json, golden, oracle_params

HARNESS = Path(__file__).resolve().parent / "kin_fast_env_harness.cu"
F32 = np.float32
PI_F = F32(np.pi)                 # 3.1415927 > pi: the joint limits +-pi as fp32
POS_TOL, ANG_TOL, EPS_BAND = 1e-5, 1e-5, 3e-6
ATAN2_TOL = 5e-7                  # 7.5e-8 fit + rcp.approx (1 ulp of t: <= 6e-8 rad) + rounding of pi/2 - r and pi - r and of the constants
MUFU_SINCOS_TOL = 2.0 ** -20.9    # sin.approx / cos.approx on [-pi, pi] (PTX ISA)


# ---- building and loading the harness ---------------------------------------------------------------------------------------------
def _nvcc_cmd(out: Path) -> list[str]:
    from rl_brain_trainer_b200 import build as kbuild

    return [kbuild._nvcc(), *kbuild.NVCC_FLAGS, "-shared", "-o", str(out), str(HARNESS)]


def compile_harness(out: Path) -> Path:
    env = dict(os.environ)
    env.pop("CC", None)   # as rl_brain_trainer_b200.build: let nvcc pick the host compiler
    env.pop("CXX", None)
    tmp = out.with_name(out.name + f".{os.getpid()}.tmp")
    r = subprocess.run(_nvcc_cmd(tmp), capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {HARNESS.name}:\n{r.stdout}{r.stderr}")
    os.replace(tmp, out)
    return out


def _harness_hash() -> str:
    from rl_brain_trainer_b200 import build as kbuild

    h = hashlib.sha256()
    for f in [HARNESS, *kbuild.source_files()]:
        h.update(f.name.encode() + b"\0" + f.read_bytes() + b"\0")
    h.update(" ".join(kbuild.NVCC_FLAGS).encode())
    return h.hexdigest()[:20]


@functools.lru_cache(maxsize=1)
def _lib() -> ctypes.CDLL:
    d = Path(tempfile.gettempdir()) / f"kin_fast_env_harness_{_harness_hash()}"
    d.mkdir(parents=True, exist_ok=True)
    so = d / "harness.so"
    if not so.exists():
        compile_harness(so)
    L = ctypes.CDLL(str(so))
    vp, i = ctypes.c_void_p, ctypes.c_int
    L.kfh_scalar.argtypes = [i, vp, vp, vp, vp, i]
    L.kfh_interp.argtypes = [vp, vp, i]
    L.kfh_fk.argtypes = [vp, i, vp, vp, i]
    L.kfh_dyn_col.argtypes = [vp]
    L.kfh_episode.argtypes = [vp, vp, i, i, i, vp, vp, vp, vp, vp, vp, i, i, vp, vp]
    return L


def _check(err: int) -> None:
    assert err == 0, f"harness launch failed: CUDA error {err}"


def _dev(a, dtype=None):
    import torch

    if a is None:
        return None
    t = torch.as_tensor(np.ascontiguousarray(a, dtype=dtype or np.float32))
    return t.cuda()


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _scalar(op: int, x, y=None):
    import torch

    x = _dev(np.asarray(x, F32))
    y = _dev(np.asarray(y, F32)) if y is not None else None
    o0, o1 = torch.empty_like(x), torch.empty_like(x)
    _check(_lib().kfh_scalar(op, _ptr(x), _ptr(y), _ptr(o0), _ptr(o1), x.numel()))
    return o0.cpu().numpy(), o1.cpu().numpy()


def _kin_params(cfg):
    from rl_brain_trainer_b200 import params

    return params.env_params(cfg)


def _fk(cfg, fast: int, q: np.ndarray) -> np.ndarray:
    import torch

    qd = _dev(np.asarray(q, F32))
    pose = torch.empty((q.shape[0], 6), dtype=torch.float32, device="cuda")
    p = _kin_params(cfg)
    _check(_lib().kfh_fk(ctypes.addressof(p), fast, _ptr(qd), _ptr(pose), q.shape[0]))
    return pose.cpu().numpy().astype(float)


@functools.lru_cache(maxsize=1)
def _dyn_cols() -> np.ndarray:
    import torch

    out = torch.zeros(36, dtype=torch.int32, device="cuda")
    _check(_lib().kfh_dyn_col(_ptr(out)))
    return out.cpu().numpy()


def _ulp(v) -> np.ndarray:
    return np.spacing(np.abs(np.asarray(v, F32))).astype(float)


def _ulp16(v) -> np.ndarray:
    a = np.abs(np.asarray(v, float))
    e = np.floor(np.log2(np.maximum(a, 2.0 ** -14)))
    return 2.0 ** (e - 10)


# ---- CPU: the harness still compiles ----------------------------------------------------------------------------------------------
def test_harness_compiles_for_sm100(tmp_path):
    """Catches harness rot (a renamed helper, a changed signature) on machines without a GPU."""
    try:
        from rl_brain_trainer_b200 import build as kbuild

        kbuild._nvcc()
    except RuntimeError:
        pytest.skip("nvcc not available")
    so = compile_harness(tmp_path / "harness.so")
    assert so.stat().st_size > 0


# ---- scalar helpers ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_atan2_fast_against_numpy():
    th = np.concatenate([np.linspace(-np.pi, np.pi, 20001), np.arange(-8, 9) * (np.pi / 4)])   # every octant, the |y| = |x| diagonals
    mags = np.concatenate([10.0 ** np.arange(-37, 31, 1.0), [2.4e-38, 3.0, 0.7]])   # 1e30 down through 1e-30 to 2 FLT_MIN
    y = (np.sin(th)[None, :] * mags[:, None]).astype(F32).ravel()
    x = (np.cos(th)[None, :] * mags[:, None]).astype(F32).ravel()
    diag = (mags[:, None] * np.array([1.0, -1.0])[None, :]).astype(F32).ravel()
    y = np.concatenate([y, diag, diag, -diag])
    x = np.concatenate([x, diag, -diag, diag])
    r, _ = _scalar(0, x, y)
    ref = np.arctan2(y.astype(float), x.astype(float))
    err = np.abs(r - ref)
    assert err.max() < ATAN2_TOL, (float(err.max()), float(x[err.argmax()]), float(y[err.argmax()]))

    # the axes and signed zeros
    m = np.array([1e30, 1.0, 1e-30, 1e-38], F32)
    z = np.zeros_like(m)
    r, _ = _scalar(0, np.concatenate([m, -m, z, z, -z, -z, -m, -m]), np.concatenate([z, z, m, -m, m, -m, z, -z]))
    k = m.size
    assert np.all(r[:k] == 0) and not np.signbit(r[:k]).any()                          # atan2(+0, x > 0) = +0
    assert np.all(r[k:2 * k] == PI_F)                                                    # atan2(+0, x < 0) = +pi
    assert np.all(r[2 * k:3 * k] == F32(np.pi / 2)) and np.all(r[3 * k:4 * k] == -F32(np.pi / 2))   # x = +0
    assert np.all(r[4 * k:5 * k] == F32(np.pi / 2)) and np.all(r[5 * k:6 * k] == -F32(np.pi / 2))   # x = -0
    assert np.all(r[6 * k:7 * k] == PI_F) and np.all(r[7 * k:8 * k] == -PI_F)            # y = +-0, x < 0: +-pi
    # both zero: atan2(+-0, +0) = +-0 like math.atan2, and atan2(+-0, -0) = +-0 where math.atan2 gives +-pi (documented)
    r, _ = _scalar(0, np.array([0.0, 0.0, -0.0, -0.0], F32), np.array([0.0, -0.0, 0.0, -0.0], F32))
    assert np.all(r == 0) and list(np.signbit(r)) == [False, True, False, True]

    # both subnormal: the ratio is not formed exactly (rcp.approx flushes), but sign and octant are right
    sub = (np.array([1e-39, 3e-40, 1e-44, 7e-41], np.float64))
    ang = np.linspace(-np.pi, np.pi, 97)
    ys = (np.sin(ang)[None, :] * sub[:, None]).astype(F32).ravel()
    xs = (np.cos(ang)[None, :] * sub[:, None]).astype(F32).ravel()
    keep = (ys != 0) & (xs != 0)
    ys, xs = ys[keep], xs[keep]
    r, _ = _scalar(0, xs, ys)
    ref = np.arctan2(ys.astype(float), xs.astype(float))
    assert np.all(np.sign(r) == np.sign(ref)) and np.all(np.abs(r - ref) <= np.pi / 4 + 1e-6)


def _sincos_inputs() -> np.ndarray:
    dense = np.linspace(-PI_F, PI_F, 1_000_001).astype(F32)
    around = []
    for k in range(-4, 5):   # +-1000 ulps around every reduction boundary k pi / 4 (quadrant and octant switches)
        c = F32(k * np.pi / 4)
        steps = np.arange(-1000, 1001)
        v = c + steps.astype(np.float64) * float(np.spacing(max(abs(c), F32(1e-6))))
        around.append(v.astype(F32))
    special = np.array([PI_F, -PI_F, np.nextafter(PI_F, F32(0)), np.nextafter(-PI_F, F32(0)), 0.0, -0.0, 1e-30, -1e-30, 1e-38, 1e-45,
                        3.1415925, -3.1415925], F32)
    x = np.concatenate([dense, *around, special])
    return x[np.abs(x) <= PI_F]


@pytest.mark.gpu
@pytest.mark.parametrize("op,name", [(1, "strict"), (2, "fast1"), (3, "mufu")])
def test_sincos_flavours_against_numpy(op, name):
    x = _sincos_inputs()
    s, c = _scalar(op, x)
    rs, rc = np.sin(x.astype(float)), np.cos(x.astype(float))
    es, ec = np.abs(s - rs), np.abs(c - rc)
    if op == 3:
        assert max(es.max(), ec.max()) <= MUFU_SINCOS_TOL, (float(es.max()), float(ec.max()))
    else:
        # a few ulp of the result (the polynomials of sinf / cosf's fast path; FAST = 1 drops the 5e-15 k term of the reduction)
        us, uc = es / _ulp(rs), ec / _ulp(rc)
        assert max(us.max(), uc.max()) <= 2.0, (name, float(us.max()), float(uc.max()), float(x[us.argmax()]), float(x[uc.argmax()]))
    tiny = np.array([0.0, 1e-30, -1e-30, 1e-38], F32)
    s, c = _scalar(op, tiny)
    if op != 3:
        assert np.array_equal(s, tiny) and np.all(c == 1.0)


@pytest.mark.gpu
def test_wrap_to_pi():
    rng = np.random.default_rng(3)
    inside = np.concatenate([rng.uniform(-3.1415925, 3.1415925, 200_000).astype(F32),
                             np.array([3.1415925, -3.1415925, 0.0, -0.0, 1e-38, -1e-45, 1.0, -2.5], F32)])
    inside = inside[np.abs(inside.astype(float)) < np.pi]
    r, _ = _scalar(4, inside)
    assert np.array_equal(r.view(np.uint32), inside.view(np.uint32)), "wrap_to_pi must return |v| < pi bit for bit"
    near = []
    for k in (-3, -2, -1, 1, 2, 3):
        c = F32(k * np.pi)
        near.append((c.astype(np.float64) + np.arange(-2000, 2001) * float(np.spacing(c))).astype(F32))
    v = np.concatenate(near)
    r, _ = _scalar(4, v)
    ref = np.mod(v.astype(float) + np.pi, 2 * np.pi) - np.pi       # pose_utils.py: floored modulo, fp64
    d = np.abs(np.mod(r - ref + np.pi, 2 * np.pi) - np.pi)         # the same angle (+pi and -pi are one point)
    # 2 pi as fp32 is 1.7e-7 off: k = 1 reduction carries that, k = 2 twice, plus the final rounding
    assert d.max() < 6e-7, float(d.max())
    # the result lies in [-pi, pi] for |v| < 2 pi (every pose-error difference); near +-3 pi the floor's argument can round up to
    # the next integer and the result lands up to 2 ulp outside
    inner = np.abs(v.astype(float)) < 2 * np.pi
    assert np.all(np.abs(r[inner]) <= PI_F) and np.all(np.abs(r) <= PI_F + 2 * np.spacing(PI_F))


@pytest.mark.gpu
def test_sqrt_and_rcp_approx():
    x = np.concatenate([10.0 ** np.linspace(-37, 37, 100_001), [1.0, 2.0, 4.0, 0.25]]).astype(F32)
    s, _ = _scalar(5, x)
    assert (np.abs(s - np.sqrt(x.astype(float))) / np.sqrt(x.astype(float))).max() < 2.0 ** -22
    r, _ = _scalar(6, x)
    assert (np.abs(r * x.astype(float) - 1.0)).max() < 2.0 ** -22
    s0, _ = _scalar(5, np.array([0.0, 1e-45], F32))   # .ftz: a subnormal counts as zero
    assert np.all(s0 == 0)


@pytest.mark.gpu
def test_interp_control_fast_against_strict():
    import torch

    rows = []
    for near, far in ((0.012, 0.06), (0.01, 0.05), (1e-4, 3.0)):
        nf, ff = F32(near), F32(far)
        pos = [0.0, nf, np.nextafter(nf, F32(0)), np.nextafter(nf, F32(1)), ff, np.nextafter(ff, F32(0)), np.nextafter(ff, F32(10)),
               2 * ff, 100.0, *np.linspace(nf, ff, 101)]
        for nv, fv in ((0.3, 1.0), (1.0, 0.2), (2.5, 2.5), (-0.7, 0.4)):
            rows += [(p, near, far, nv, fv, 0.77) for p in pos]
    degenerate = [(p, near, far, 0.3, 1.0, 0.77) for p in (0.0, 0.02, 1.0) for near, far in ((0.05, 0.05), (0.05, 0.01), (0.0, 0.1), (-0.1, 0.1))]
    a = np.array(rows + degenerate, F32)
    out = torch.empty((a.shape[0], 2), dtype=torch.float32, device="cuda")
    ad = _dev(a)
    _check(_lib().kfh_interp(_ptr(ad), _ptr(out), a.shape[0]))
    o = out.cpu().numpy()
    strict, fast = o[:, 0], o[:, 1]
    pos, near, far, nv, fv, fb = (a[:, i] for i in range(6))
    deg = (near <= 0) | (far <= near)
    assert np.all(strict[deg] == fb[deg]) and np.all(fast[deg] == fb[deg]), "degenerate thresholds must return the fallback"
    ok = ~deg
    lo, hi = ok & (pos <= near), ok & (pos >= far)
    assert np.all(strict[lo] == nv[lo]) and np.all(fast[lo] == nv[lo])     # alpha = 0 exactly
    assert np.all(strict[hi] == fv[hi])
    # the fast form has no endpoint branch: at pos >= far, alpha = (far - near) * rcp(far - near) may be 1 - 2^-24 and far - near is
    # rounded, so the result is far_v to 1 ulp of max(|near_v|, |far_v|)
    scale = _ulp(np.maximum(np.abs(nv), np.abs(fv)))
    assert np.all(np.abs(fast[hi] - fv[hi]) <= scale[hi])
    mid = ok & ~lo & ~hi
    assert np.all(np.abs(fast[mid] - strict[mid]) <= 3 * scale[mid])
    ref = nv + (pos.astype(float) - near) / (far.astype(float) - near) * (fv.astype(float) - nv)
    assert np.all(np.abs(fast[mid] - ref[mid]) <= 4 * scale[mid] + 1e-9)


# ---- forward kinematics -----------------------------------------------------------------------------------------------------------
def _geo_err(pose, ref):
    """Geodesic angle between the rotations rebuilt from the two Euler triples.  Within 1 % of gimbal lock (|cos pitch| < 1e-2) roll
    and yaw each carry ~1e-7 / cos(pitch) of fp32 rounding -- the strict flavour too -- and the rebuilt rotation inherits it: the
    bound is scaled there like the Euler components' (4e-3 gives 2e-5 rad)."""
    return (_geodesic(pose[:, 3:], ref[:, 3:]) * np.minimum(1.0, np.abs(np.cos(ref[:, 4])) / 1e-2)).max()


def _euler_err(pose, ref):
    d = np.abs((pose[:, 3:] - ref[:, 3:] + np.pi) % (2 * np.pi) - np.pi)
    return (d * np.maximum(np.abs(np.cos(ref[:, 4:5])), 1e-4)).max()


@functools.lru_cache(maxsize=1)
def _fk_inputs() -> dict[str, np.ndarray]:
    cfg = env_config("approach_dynamic_scale_big")
    lo = np.array([s.lower for s in cfg.joint_specs]).astype(F32)
    hi = np.array([s.upper for s in cfg.joint_specs]).astype(F32)
    rng = np.random.default_rng(17)
    rand = rng.uniform(lo, hi, (4096, 7)).astype(F32)
    at_lim = np.where(rng.random((1024, 7)) < 0.5, lo, hi).astype(F32)
    at_lim[:512] = np.where(rng.random((512, 7)) < 0.5, at_lim[:512], rand[:512])
    pool = rng.uniform(lo, hi, (60_000, 7)).astype(F32)
    pp = ko.fk_pose6(pool.astype(float))
    pick = lambda score: pool[np.argsort(score)[:256]]  # noqa: E731
    # near roll / yaw = +-pi and near pitch = +-pi/2 (down to |cos pitch| = 1e-3; at exact gimbal lock roll and yaw are undetermined)
    ok = np.abs(np.cos(pp[:, 4])) >= 1e-3
    gap = lambda v: np.where(ok, v, np.inf)  # noqa: E731
    near_pi = np.concatenate([pick(gap(np.pi - np.abs(pp[:, 3]))), pick(gap(np.pi - np.abs(pp[:, 5]))),
                              pick(gap(np.abs(np.abs(pp[:, 4]) - np.pi / 2)))])
    return {"golden": golden("fk.npz")["q"].astype(F32), "random": rand, "limits": at_lim, "euler_edges": near_pi}


@pytest.mark.gpu
@pytest.mark.parametrize("fast", [0, 1, 2])
def test_fk_flavours_match_oracle(fast):
    cfg = env_config("approach_dynamic_scale_big")
    worst = {}
    for name, q in _fk_inputs().items():
        ref = ko.fk_pose6(q.astype(float))
        pose = _fk(cfg, fast, q)
        assert np.abs(pose[:, :3] - ref[:, :3]).max() < POS_TOL, name
        assert _geo_err(pose, ref) < ANG_TOL, name
        assert _euler_err(pose, ref) < ANG_TOL, name
        if fast:
            strict = _fk(cfg, 0, q)
            dp = np.abs(pose[:, :3] - strict[:, :3]).max()
            da = max(_geo_err(pose, strict), _euler_err(pose, strict))
            worst[name] = (float(dp), float(da))
            # from the primitives: a sine / cosine pair with error e perturbs a joint rotation by <= sqrt(2) e (2-norm), seven of
            # them move the tip by <= 7 sqrt(2) e x reach (1.07 m) and the rotation entries by <= 7 sqrt(2) e.  e = 2 ulp (FAST = 1)
            # or 2^-20.9 (FAST = 2).  The Euler angles add the atan2_fast error and their conditioning near pitch +-pi/2: FAST = 1
            # stays within 2e-6 rad of the strict flavour, FAST = 2 within the 1e-5 rad pose tolerance (8.7e-6 near pitch +-pi/2)
            e = 2 * 2.0 ** -23 if fast == 1 else MUFU_SINCOS_TOL
            assert dp < 7 * np.sqrt(2) * e * 1.07 + 1e-7, (name, dp)
            assert da < (2e-6 if fast == 1 else ANG_TOL), (name, da)
    print(f"FAST={fast} vs strict FK, max |d pos| / max angle:", worst)


# ---- episodes: reset, prime, T steps, against the oracle step by step ------------------------------------------------------------
REC_Q, REC_DQ, REC_PA, REC_POSE, REC_PE, REC_OE = slice(0, 7), slice(7, 14), slice(14, 21), slice(21, 27), slice(27, 30), slice(30, 33)
REC_POS, REC_ORI, REC_RPOS, REC_RORI, REC_MARGIN, REC_QN = 33, 34, 35, 36, slice(37, 44), slice(44, 51)
REC_REWARD, REC_MINPOS, REC_OBS = 51, 52, slice(56, 112)


def _gpu_episode(cfg, cfg2, fast, mode, handoff, ep, actions):
    import torch

    n, T = ep["iq"].shape[0], actions.shape[0]
    rec = torch.zeros((T + 2, n, 112), dtype=torch.float32, device="cuda")
    irec = torch.zeros((T + 2, n, 8), dtype=torch.int32, device="cuda")
    p1, p2 = _kin_params(cfg), _kin_params(cfg2)
    bufs = {k: _dev(ep.get(k)) for k in ("iq", "idq", "ipa", "gq", "gp")}
    act = _dev(np.asarray(actions, F32))
    _check(_lib().kfh_episode(ctypes.addressof(p1), ctypes.addressof(p2), fast, mode, handoff, *(_ptr(bufs[k]) for k in ("iq", "idq", "ipa", "gq", "gp")),
                              _ptr(act), T, n, _ptr(rec), _ptr(irec)))
    return rec.cpu().numpy().astype(float), irec.cpu().numpy()


class _Oracle:
    """n oracle envs in lock-step (fp64), with structured views of the C arrays."""

    def __init__(self, cfg, n):
        self.params, self.n = oracle_params(cfg), n
        self.states = ko.state_array(n)

    def reset(self, mode, iq, gq, gp=None, idq=None, ipa=None, params=None):
        L = ko.lib()
        params = params or self.params
        f = lambda a, e: None if a is None else ko._dptr(np.ascontiguousarray(a[e], dtype=np.float64))  # noqa: E731
        for e in range(self.n):
            L.kor_reset(ctypes.byref(params), ctypes.byref(self.states[e]), mode, f(iq, e), f(idq, e), f(ipa, e), f(gq, e), f(gp, e))

    def view(self):
        return np.frombuffer(self.states, dtype=np.dtype(ko.State)).copy()

    def obs(self, params=None):
        out = np.zeros((self.n, 56), F32)
        for e in range(self.n):
            ko.lib().kor_observation(ctypes.byref(params or self.params), ctypes.byref(self.states[e]), ko._fptr(out[e]))
        return out


def _oracle_episode(cfg, cfg2, mode, handoff, ep, actions):
    """The oracle's view of every record row (row 0 = after reset, T + 1 = after the handoff's re-reset)."""
    n, T = ep["iq"].shape[0], actions.shape[0]
    f64 = lambda k: None if ep.get(k) is None else np.asarray(ep[k], F32).astype(float)  # noqa: E731
    orc = _Oracle(cfg, n)
    p2 = oracle_params(cfg2)
    orc.reset(mode, f64("iq"), f64("gq"), f64("gp"), f64("idq"), f64("ipa"))
    rows = [None] * (T + 2)
    st = orc.view()
    rows[0] = {"st": st, "obs": orc.obs(), "pos": st["entry_position_error_norm"], "ori": st["entry_orientation_error_norm"], "out": None}
    params = orc.params
    for t in range(1, T + 1):
        robs, routs = ko.step_batch(params, orc.states, np.asarray(actions[t - 1], F32).astype(float))
        out = np.frombuffer(routs, dtype=np.dtype(ko.StepOut)).copy()
        rows[t] = {"st": orc.view(), "obs": robs, "pos": out["position_error_norm"], "ori": out["orientation_error_norm"], "out": out}
        if t == handoff:
            s = rows[t]["st"]
            params = p2
            orc.reset(1, s["q"], s["goal_q"], s["goal_pose6"], s["dq"], s["prev_action"], params=p2)
            st = orc.view()
            rows[T + 1] = {"st": st, "obs": orc.obs(p2), "pos": st["entry_position_error_norm"], "ori": st["entry_orientation_error_norm"], "out": None}
    return rows


def _folded_columns_hold_constants(obs: np.ndarray, mode: int) -> None:
    """The 20 observation columns tc16::load_weights folds into the layer-1 bias hold exactly those constants."""
    const = np.zeros(56)
    const[20 + mode] = 1.0
    const[47] = 1.0
    dyn = set(_dyn_cols().tolist())
    folded = [c for c in range(56) if c not in dyn]
    assert len(folded) == 20
    assert np.array_equal(obs[:, folded], np.broadcast_to(const[folded], (obs.shape[0], 20))), f"folded columns differ (mode {mode})"


def _state_tol(cfg, mode) -> float:
    """5e-6 (test_gpu_env_parity) -- except in dock mode with a dynamic action limit: the limit and the dq-change scale follow the
    previous position error through the interpolation (slopes of ~50 / m in these configs), so a 1e-6 m difference in the pose error
    moves the clipped command, and the difference accumulates over the episode."""
    dyn = cfg.dock_dynamic_action_limit_far_pos_threshold_m > cfg.dock_dynamic_action_limit_near_pos_threshold_m > 0
    return 5e-5 if (mode == 1 and dyn) else 5e-6


def _compare_episode(cfg, cfg2, fast, mode, handoff, ep, actions, ref):
    rec, irec = _gpu_episode(cfg, cfg2, fast, mode, handoff, ep, actions)
    n, T = ep["iq"].shape[0], actions.shape[0]
    dyn = _dyn_cols()
    pos_thr, ori_thr, act_thr, dq_thr = (np.union1d(a, b) for a, b in zip(_thresholds(cfg), _thresholds(cfg2)))
    clean = np.ones(n, dtype=bool)
    stats = {"max_q": 0.0, "max_pose": 0.0, "max_reward": 0.0, "max_obs": 0.0, "checked": 0}
    state_tol = max(_state_tol(cfg, mode), _state_tol(cfg2, 1) if handoff else 0.0)
    # FAST = 2's MUFU sine / cosine move the pose error norms by up to ~1e-6 (Euler angles up to 9e-6 rad off the strict ones near
    # pitch +-pi/2); the progress terms weigh that into the reward
    reward_tol = 5e-4 if fast == 2 else 2e-4
    order = [0, *range(1, T + 1)]
    if 0 < handoff < T:
        order.insert(handoff + 1, T + 1)
    prev_pos, prev_ori = ref[0]["pos"], ref[0]["ori"]
    cur_mode = mode
    for t in order:
        r, ir, R = rec[t], irec[t], ref[t]
        st = R["st"]
        if t == T + 1:
            cur_mode = 1
            prev_pos, prev_ori = R["pos"], R["ori"]
        _folded_columns_hold_constants(R["obs"], cur_mode)
        # kinematic state and pose: every episode, every row
        dq_max = max(np.abs(r[:, REC_Q] - st["q"]).max(), np.abs(r[:, REC_DQ] - st["dq"]).max(), np.abs(r[:, REC_PA] - st["prev_action"]).max())
        assert dq_max < state_tol, (t, dq_max)
        pose, rpose = r[:, REC_POSE], st["ee_pose6"]
        assert np.abs(pose[:, :3] - rpose[:, :3]).max() < POS_TOL, t
        ang = max(_geo_err(pose, rpose), _euler_err(pose, rpose))
        assert ang < ANG_TOL, (t, ang)
        stats["max_q"], stats["max_pose"] = max(stats["max_q"], dq_max), max(stats["max_pose"], ang)
        assert np.abs(r[:, REC_POS] - R["pos"]).max() < POS_TOL, t
        cond = np.maximum(np.minimum(np.abs(np.cos(rpose[:, 4])), np.abs(np.cos(st["goal_pose6"][:, 4]))), 1e-4)
        assert (np.abs(r[:, REC_ORI] - R["ori"]) * cond).max() < 2 * ANG_TOL, t
        # the carried norms are the norms of this row's pose (after reset and after the handoff too), the margins / normalised q in range
        for c, rc in ((REC_POS, REC_RPOS), (REC_ORI, REC_RORI)):
            bad = np.abs(r[:, c] - r[:, rc]) > 2 * _ulp(r[:, rc])
            assert not bad.any(), f"row {t}: carried norm {c} is not the norm of the pose (env {int(np.argmax(bad))})"
        m = r[:, REC_MARGIN]
        assert m.min() >= 0.0 and m.max() <= 1.0, (t, m.min(), m.max())
        if fast:
            qn = r[:, REC_QN]
            assert qn.min() >= -1.0 and qn.max() <= 1.0, (t, qn.min(), qn.max())
        # discrete outcomes and rewards: episodes with no epsilon-band event so far
        if R["out"] is not None:
            o = R["out"]
            band = _near(R["pos"], pos_thr, EPS_BAND) | _near(R["ori"], ori_thr, 4 * EPS_BAND) | _near(o["action_l2"], act_thr, EPS_BAND) \
                | _near(o["executed_delta_q_l2"], dq_thr, EPS_BAND / 3)
            band |= (np.abs(R["pos"] - prev_pos) < EPS_BAND / 3) | (np.abs(R["ori"] - prev_ori) < EPS_BAND)
            prev_pos, prev_ori = R["pos"], R["ori"]
            clean &= ~band
            d = ir[:, 0]
            g_flags = np.stack([d & 1, (d >> 1) & 1, (d >> 2) & 1, (d >> 3) & 1, (d >> 4) & 1, (d >> 5) & 3], 1)
            r_flags = np.stack([o["terminated"], o["truncated"], o["success"], o["curr_in_pre_near_goal"], o["curr_in_near_goal"], o["reason"]], 1)
            assert np.array_equal(g_flags[clean], r_flags[clean]), f"flags differ at step {t}"
            fl = ir[:, 5]
            g_cnt = np.stack([ir[:, 1], ir[:, 2], ir[:, 3], ir[:, 4], fl & 1, (fl >> 1) & 1], 1)
            r_cnt = np.stack([st["episode_step"], st["dwell_count"], st["near_goal_entry_count"], st["near_goal_drift_count"],
                              st["pre_near_goal_hit"], st["near_goal_hit"]], 1)
            assert np.array_equal(g_cnt[clean], r_cnt[clean]), f"counters differ at step {t}"
            err = np.abs(r[:, REC_REWARD] - o["reward"]) / np.maximum(1.0, np.abs(o["reward"]))
            assert (err[clean] < reward_tol).all(), f"reward differs at step {t}: {float(err[clean].max())}"
            stats["max_reward"] = max(stats["max_reward"], float(err[clean].max(initial=0.0)))
            assert np.abs(r[clean, REC_MINPOS] - st["min_pos_error"][clean]).max(initial=0.0) < POS_TOL
            stats["checked"] += int(clean.sum())
        robs = R["obs"].astype(float)
        if fast:
            # each obs_pack column k is the oracle's column dyn_col(k) to fp16 rounding (+ the fp32 state's own error)
            got, want = r[:, REC_OBS][:, :36], robs[:, dyn]
            tol = 0.5 * _ulp16(np.maximum(np.abs(got), np.abs(want))) + 5e-5
            bad = np.abs(got - want) > tol
            bad[~clean] = False
            assert not bad.any(), f"row {t}: obs_pack column {int(np.argwhere(bad)[0][1])} differs from the oracle observation"
            stats["max_obs"] = max(stats["max_obs"], float((np.abs(got - want) - 0.5 * _ulp16(want))[clean].max(initial=0.0)))
        else:
            d = np.abs(r[:, REC_OBS] - robs)[clean]
            assert d.max(initial=0.0) < 5e-5, (t, float(d.max()))
            stats["max_obs"] = max(stats["max_obs"], float(d.max(initial=0.0)))
    return stats


# ---- episode inputs ---------------------------------------------------------------------------------------------------------------
def _trace_case(fixture, preset, mode):
    trace = golden(fixture)
    cfg = env_config_from_json(GOLD / preset) if preset.endswith(".json") else env_config(preset)
    starts = trace["episode_start"]
    n = len(starts) - 1
    T = int(np.max(np.diff(starts)))
    actions = np.zeros((T, n, 7))
    for e in range(n):
        seg = trace["action"][starts[e]:starts[e + 1]]
        actions[: len(seg), e] = seg
    has_gp = trace["reset_has_goal_pose6"].astype(bool)
    ep = {"iq": trace["reset_initial_q"], "gq": trace["reset_goal_q"], "gp": trace["reset_goal_pose6"] if has_gp.all() else None,
          "idq": trace["reset_initial_dq"], "ipa": trace["reset_initial_prev_action"]}
    return cfg, cfg, mode, 0, ep, actions


def _random_case(preset, mode, scale):
    """The random open-loop batches of test_gpu_env_parity.test_random_batch_open_loop."""
    cfg = env_config(preset)
    rng = np.random.default_rng(11 + mode)
    n, T = 2048, 48
    stages = env_config("approach_dynamic_scale_big").curriculum_config.stages
    st = [stages[i % len(stages)] for i in range(n)]
    gq = np.array([np.asarray(s.goal_q) + rng.uniform(-1, 1, 7) * np.asarray(s.goal_noise) for s in st])
    if mode == 0:
        iq = np.array([np.asarray(s.start_q) + rng.uniform(-1, 1, 7) * np.asarray(s.start_noise) for s in st])
        actions = np.zeros((T, n, 7))
        q = iq.copy()
        dl = np.array([sp.delta_limit for sp in cfg.joint_specs]) * cfg.action_delta_scale
        for t in range(T):
            a = np.clip((gq - q) / dl * 0.6 + rng.normal(0, 0.05, (n, 7)) * (rng.random((n, 1)) < 0.5), -1.3, 1.3)
            actions[t] = a
            q = q + np.clip(a, -1, 1) * dl
    else:
        iq = gq + rng.uniform(-0.003, 0.003, (n, 7))
        actions = rng.normal(0, 1.0, (T, n, 7)) * scale * rng.choice([0.1, 1.0, 4.0], size=(1, n, 1))
    ep = {"iq": iq, "gq": gq, "idq": rng.uniform(-0.001, 0.001, (n, 7)), "ipa": rng.uniform(-0.05, 0.05, (n, 7))}
    return cfg, cfg, mode, 0, ep, actions


def _saturating_case(cfg, seed, n=512, T=64):
    """+-1 action tapes that drive joints into their limits and hold them there for many steps."""
    rng = np.random.default_rng(seed)
    lo = np.array([s.lower for s in cfg.joint_specs])
    hi = np.array([s.upper for s in cfg.joint_specs])
    dl = np.array([s.delta_limit for s in cfg.joint_specs]) * cfg.action_delta_scale
    side = rng.choice([-1.0, 1.0], (n, 7))
    iq = np.where(side > 0, hi, lo) - side * dl * rng.uniform(0, 12, (n, 7))          # within a dozen steps of a limit
    iq[: n // 8] = np.where(side[: n // 8] > 0, hi, lo)                                  # some start exactly at it
    gq = np.clip(iq + rng.uniform(-0.2, 0.2, (n, 7)), lo, hi)
    actions = np.broadcast_to(side * 1.0, (T, n, 7)).copy()
    flip = rng.random((T, n, 7)) < 0.03                                                   # brief excursions off the limit
    actions[flip] *= -1.0
    actions[:, : n // 4] *= rng.uniform(1.0, 3.0, (1, n // 4, 7))                         # beyond +-1: the step clips
    return {"iq": iq, "gq": gq}, actions


def _saturating_limits_case():
    cfg = env_config("approach_dynamic_scale_big")
    ep, actions = _saturating_case(cfg, 21)
    return cfg, cfg, 0, 0, ep, actions


def _custom_limits_cfg(seed):
    """Random asymmetric joint limits whose spans are not representable (kin_params_create accepts any lower < upper)."""
    cfg = env_config("approach_dynamic_scale_big")
    rng = np.random.default_rng(seed)
    specs = []
    for i, s in enumerate(cfg.joint_specs):
        lo = rng.uniform(-3.0, 1.0)
        hi = lo + rng.choice([rng.uniform(0.05, 0.2), rng.uniform(0.3, 3.0)])
        specs.append(replace(s, lower=float(lo), upper=float(hi), delta_limit=float(min(s.delta_limit, 0.25 * (hi - lo) / cfg.action_delta_scale))))
    return replace(cfg, joint_specs=type(cfg.joint_specs)(specs))


def _custom_limits_case(seed):
    cfg = _custom_limits_cfg(seed)
    ep, actions = _saturating_case(cfg, seed, n=512, T=48)
    return cfg, cfg, 0, 0, ep, actions


def _wrap_case():
    """Explicit goals with roll / yaw near +-pi: the orientation error crosses the wrap while the arm moves."""
    cfg = env_config("approach_dynamic_scale_big")
    rng = np.random.default_rng(31)
    q = _fk_inputs()["euler_edges"][:512].astype(float)
    pose = ko.fk_pose6(q)
    gp = pose.copy()
    shift = rng.uniform(-0.03, 0.03, (q.shape[0], 2))
    gp[:, 3] = (pose[:, 3] + shift[:, 0] + np.pi) % (2 * np.pi) - np.pi
    gp[:, 5] = (pose[:, 5] + shift[:, 1] + np.pi) % (2 * np.pi) - np.pi
    gp[::2, 3] = np.sign(gp[::2, 3]) * (np.pi - rng.uniform(0, 2e-3, gp[::2, 3].shape))   # right at the seam
    gp[:, :3] += rng.uniform(-0.01, 0.01, (q.shape[0], 3))
    actions = rng.normal(0, 0.3, (40, q.shape[0], 7))
    return cfg, cfg, 0, 0, {"iq": q, "gq": q, "gp": gp}, actions


def _dock_dynamic_cfg():
    cfg = env_config("finisher_noop_ft")
    return replace(cfg, dock_dynamic_action_limit_near_pos_threshold_m=0.01, dock_dynamic_action_limit_far_pos_threshold_m=0.04,
                   dock_dynamic_residual_action_limit_near=0.25, dock_dynamic_residual_action_limit_far=0.9,
                   dock_dynamic_delta_q_change_limit_scale_near=0.3, dock_dynamic_delta_q_change_limit_scale_far=0.8, dock_action_delta_scale=0.05)


def _dock_dynamic_case():
    """Dock episodes whose previous position error sweeps across the near / far thresholds of the dynamic action limit."""
    cfg = _dock_dynamic_cfg()
    rng = np.random.default_rng(41)
    n, T = 1024, 40
    gq = rng.uniform(-0.4, 0.4, (n, 7))
    iq = gq + rng.uniform(-1, 1, (n, 7)) * rng.choice([0.002, 0.01, 0.03, 0.06], (n, 1))
    # a proportional controller towards the goal with noise: the error shrinks through the band, then jitters around the near threshold
    actions = np.zeros((T, n, 7))
    q = iq.copy()
    dl = np.array([s.delta_limit for s in cfg.joint_specs]) * cfg.dock_action_delta_scale
    for t in range(T):
        a = np.clip((gq - q) / dl * 0.3 + rng.normal(0, 0.3, (n, 7)), -1.5, 1.5)
        actions[t] = a
        q = q + np.clip(a, -1, 1) * dl * 0.5
    return cfg, cfg, 1, 0, {"iq": iq, "gq": gq, "idq": rng.uniform(-0.002, 0.002, (n, 7))}, actions


def _handoff_case():
    """Approach episodes re-reset in dock mode with the finisher's parameters after step 24, as the rollout's handoff does."""
    acfg, fcfg = env_config("approach_dynamic_scale_big"), env_config("finisher_noop_ft")
    _, _, _, _, ep, actions = _random_case("approach_dynamic_scale_big", 0, 1.0)
    return acfg, fcfg, 0, 24, {k: v[:1024] for k, v in ep.items()}, actions[:, :1024]


CASES = {
    "trace_approach": lambda: _trace_case("trace_approach.npz", "approach_dynamic_scale_big", 0),
    "trace_dock": lambda: _trace_case("trace_dock.npz", "finisher_noop_ft", 1),
    "trace_dock_alt": lambda: _trace_case("trace_dock_alt.npz", "trace_dock_alt_config.json", 1),
    "trace_approach_alt": lambda: _trace_case("trace_approach_alt.npz", "trace_approach_alt_config.json", 0),
    "random_approach": lambda: _random_case("approach_dynamic_scale_big", 0, 1.0),
    "random_dock": lambda: _random_case("finisher_noop_ft", 1, 0.05),
    "saturating_limits": _saturating_limits_case,
    "euler_wrap_goals": _wrap_case,
    "dock_dynamic_limits": _dock_dynamic_case,
    "custom_limits_a": lambda: _custom_limits_case(51),
    "custom_limits_b": lambda: _custom_limits_case(52),
    "handoff": _handoff_case,
}


@functools.lru_cache(maxsize=2)
def _case_with_reference(name):
    cfg, cfg2, mode, handoff, ep, actions = CASES[name]()
    ep = {k: (None if v is None else np.asarray(v, F32)) for k, v in ep.items()}
    actions = np.asarray(actions, F32)
    return cfg, cfg2, mode, handoff, ep, actions, _oracle_episode(cfg, cfg2, mode, handoff, ep, actions)


@pytest.mark.gpu
@pytest.mark.parametrize("fast", [0, 1, 2])
@pytest.mark.parametrize("case", list(CASES))
def test_episode_steps_match_oracle(case, fast):
    cfg, cfg2, mode, handoff, ep, actions, ref = _case_with_reference(case)
    stats = _compare_episode(cfg, cfg2, fast, mode, handoff, ep, actions, ref)
    n, T = ep["iq"].shape[0], actions.shape[0]
    # joints held at their limits leave the pose unchanged from step to step: "curr < prev" is then undecidable and the band
    # takes those episodes out of the flag / counter / reward comparison
    assert stats["checked"] > (0.05 if case.startswith(("saturating", "custom")) else 0.2) * n * T, stats
    print(case, f"FAST={fast}", stats)


@pytest.mark.gpu
def test_custom_limits_reach_the_qn_rounding_edge():
    """The custom-limit cases do exercise the rounding the qn clamp exists for: 2 k_inv_span (hi - lo) > 1 in fp32 for some joint."""
    hits = 0
    for seed in (51, 52):
        p = _kin_params(_custom_limits_cfg(seed))
        for i in range(7):
            lo, hi, inv = F32(p.joint_lower[i]), F32(p.joint_upper[i]), F32(p.k_inv_span[i])
            hits += int(F32(np.float64(F32(2) * inv) * np.float64(F32(hi - lo)) - 1.0) > 1.0)
    assert hits > 0
