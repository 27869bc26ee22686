"""CPU-only: the C-ABI library loads and exports every symbol include/lanpaint_b200.h
declares, its structs have the documented layout, and the host-side logic (coefficient
table, schedule) agrees with the oracle.  No device calls here."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from lanpaint_b200 import _native, schedule
from oracle import langevin_oracle as O


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "lanpaint_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _native.load()
    declared = _declared_symbols()
    assert len(declared) >= 12
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert sorted(_native.SYMBOLS) == declared, "binding list and header drifted apart"
    assert lib.lp_abi_version() == _native.ABI_VERSION == 6


def test_struct_layouts_match_header():
    assert C.sizeof(_native.Hyper) == 40
    assert C.sizeof(_native.Dims) == 48
    assert C.sizeof(_native.Rng) == 56
    assert C.sizeof(_native.Heads) == 32 and _native.Heads.dtype.offset == 16 and _native.Heads.cfg.offset == 24
    assert _native.Rng.seed.offset == 24 and _native.Rng.state.offset == 48
    assert _native.TABLE_STRIDE == 32


def test_index_math_selftest():
    """multiply-shift division used for (row, channel, site) decomposition is exact for every n < 2^31"""
    assert _native.load().lp_selftest_index_math(2_000_000) == 0


def test_status_strings():
    lib = _native.load()
    assert lib.lp_status_string(0) == b"ok"
    assert b"invalid" in lib.lp_status_string(1)
    with pytest.raises(_native.NativeError):
        _native.check(1, "unit")


def test_build_table_rejects_null():
    lib = _native.load()
    assert lib.lp_build_coef_table(None, None, None, None, None, 1, None, None) == 1


def _oracle_table_row(abt32: float, ve32: float, hp: O.Hyper):
    """The same quantities from the oracle's (reference-ordered) tensor code, in fp64."""
    abt = torch.tensor([abt32], dtype=torch.float64)
    step = hp.step_size * (1 - abt).clamp(min=hp.min_step_frac)
    cf = O.branch_coefficients(abt, step, abt ** 0, hp.beta * abt ** 0, hp.lam)
    rows = {}
    for k, (A, dt) in enumerate(((cf.A_x, cf.half_dt_x), (cf.A_y, cf.half_dt_y))):
        for tag, h in (("f", dt), ("h", dt / 2)):
            # feed ou_advance unit impulses to read e, k, sd back out of the reference formula
            e = O.ou_advance(torch.ones(1, dtype=torch.float64), h, A, torch.zeros(1, dtype=torch.float64), cf.D_x,
                             lambda t: torch.zeros_like(t))
            kk = O.ou_advance(torch.zeros(1, dtype=torch.float64), h, A, torch.ones(1, dtype=torch.float64), cf.D_x,
                              lambda t: torch.zeros_like(t))
            sd = O.ou_advance(torch.zeros(1, dtype=torch.float64), h, A, torch.zeros(1, dtype=torch.float64), cf.D_x,
                              lambda t: torch.ones_like(t))
            rows[(k, tag)] = (float(e), float(kk), float(sd))
        rows[(k, "A")] = float(A)
        rows[(k, "dt")] = float(dt)
    return rows


@pytest.mark.parametrize("flow", [False, True])
@pytest.mark.parametrize("sigma", [0.0292, 0.3, 1.0, 2.0, 14.6146])
@pytest.mark.parametrize("min_frac,lam,beta,step", [(1.0, 5.0, 1.0, 0.2), (0.0, 8.0, 1.5, 0.15), (0.4, 0.1, 1.0, 1.0)])
def test_coef_table_matches_oracle_formulas(flow, sigma, min_frac, lam, beta, step):
    if flow:
        sigma = min(sigma / 15.0 + 0.01, 0.99)
    s = torch.tensor([sigma], dtype=torch.float32)
    ve, abt, _ = schedule.times_from_sigma(s, flow)
    ve_o, abt_o, _ = O.times_from_sigma(s, flow)
    assert torch.equal(ve, ve_o) and torch.equal(abt, abt_o)
    hp = schedule.Hyper(step, lam, beta, min_frac, flow)
    tab = schedule.build_table(abt.numpy(), ve.numpy(), hp, rep_noise=[sigma], rep_y=[1.0 - sigma])[0]
    ohp = O.Hyper(lam=lam, beta=beta, step_size=step, min_step_frac=min_frac, flow=flow)
    want = _oracle_table_row(float(abt), float(ve), ohp)
    a = float(abt)
    inv1m = 1.0 / (1.0 - a)
    close = lambda got, ref: abs(got - ref) <= 2e-7 * max(1e-30, abs(ref)) + 1e-38
    assert close(tab[0], np.sqrt(a) * inv1m)
    S = 1.0 / (np.sqrt(a) + np.sqrt(1 - a)) if flow else np.sqrt(1 + float(ve) ** 2)
    assert close(tab[1], S) and close(tab[2], 1 / S)
    assert close(tab[3], lam) and close(tab[4], 1 + lam) and close(tab[5], sigma) and close(tab[6], 1 - sigma)
    assert tab[7] == 1.0
    for k in (0, 1):
        c = tab[8 + 8 * k: 16 + 8 * k]
        assert close(c[0], want[(k, "A")] - inv1m) or abs(c[0]) < 1e-30
        assert close(c[1], want[(k, "dt")])
        for j, tag in ((2, "f"), (5, "h")):
            e, kk, sd = want[(k, tag)]
            assert close(c[j], e) and close(c[j + 1], kk) and close(c[j + 2], sd), (k, tag, c[j:j + 3], (e, kk, sd))


def test_times_from_sigma_is_bit_identical_to_oracle():
    for flow in (False, True):
        s = torch.rand(64) * (0.98 if flow else 14.0) + 0.01
        for a, b in zip(schedule.times_from_sigma(s, flow), O.times_from_sigma(s, flow)):
            assert torch.equal(a, b)


def test_effective_inner_steps_matches_reference_wrapper_logic():
    sig = O.karras_sigmas(20)
    host = [float(v) for v in sig]
    for n in (0, 1, 5, 10):
        for i in range(20):
            s = sig[i] * torch.ones(2)
            tm = O.times_from_sigma(s, False)
            want = O.inner_steps_for(s, sig, tm.abt, n)
            got = schedule.effective_inner_steps(n, host, float(torch.mean(s)), float((1.0 - tm.abt).mean()))
            assert got == want, (n, i)
    assert schedule.min_step_frac_effective_steps(5, 0.025, 0.05) == 2
    assert schedule.min_step_frac_effective_steps(5, 0.005, 0.05) == 0


def test_engine_requires_the_native_library(monkeypatch):
    """No silent fallback: with the .so gone the engine cannot even be constructed."""
    monkeypatch.setattr(_native, "_lib", None)
    monkeypatch.setattr(_native, "_LIB_PATH", "/nonexistent/liblanpaint_b200.so")
    from lanpaint_b200.engine import LanPaint
    with pytest.raises(_native.NativeError):
        LanPaint(object(), 5, 15.0, 5.0, 1.0, 0.2)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "lanpaint_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cc", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


def test_oversized_and_malformed_geometry_is_refused_before_any_launch():
    """>= 2^31 elements is outside the 32-bit index arithmetic: the ABI says so (LP_ERR_UNSUPPORTED) instead of
    wrapping around; inconsistent dims are LP_ERR_INVALID.  Both are decided before any CUDA call."""
    lib = _native.load()
    P = C.c_void_p
    fake = P(0x1000)  # never dereferenced: validation fails first
    big = _native.Dims(1 << 20, 4096, 1024, 4096, 1024, 0)          # 2^32 elements
    assert lib.lp_prologue_f32(fake, fake, fake, fake, fake, None, fake, C.byref(big), None) == 4
    assert lib.lp_epilogue_f32(fake, fake, fake, fake, C.byref(big), None) == 4
    r = _native.Rng(mode=_native.RNG_PHILOX)
    assert lib.lp_substep_f32(fake, fake, fake, fake, fake, fake, None, None, fake, C.byref(big), C.byref(r), 3, None) == 4
    bad = _native.Dims(2, 100, 30, 100, 0, 0)                        # per_row not a multiple of spatial
    assert lib.lp_epilogue_f32(fake, fake, fake, fake, C.byref(bad), None) == 1
    neg = _native.Dims(2, 64, 16, 64, 16, 80)                        # row_split beyond the row
    assert lib.lp_epilogue_f32(fake, fake, fake, fake, C.byref(neg), None) == 1
    empty = _native.Dims(0, 64, 16, 64, 16, 0)                       # empty batch: a no-op that succeeds
    assert lib.lp_epilogue_f32(fake, fake, fake, fake, C.byref(empty), None) == 0
    assert lib.lp_substep_f32(fake, fake, fake, fake, fake, fake, None, None, fake, C.byref(empty), C.byref(r), 9, None) == 1
    for name in (b"no-such-option", b"tma_boundary", b"tma_min"):
        assert lib.lp_set_option(name, 1) == 1, name


def test_host_schedule_reproduces_the_reference_step_counts():
    """runner.HostSchedule (the sync-free schedule of SURVEY 8f rank 3) against the oracle's per-step logic."""
    from lanpaint_b200.runner import HostSchedule, karras_sigmas
    ks = karras_sigmas(20)
    assert torch.allclose(torch.tensor(ks), O.karras_sigmas(20), rtol=0, atol=0)
    for n, subs, calls in ((5, 53, 73), (10, 106, 126), (0, 0, 20)):
        sched = HostSchedule(ks, batch=3, n_inner=n)
        assert (sched.substeps, sched.model_calls) == (subs, calls)
        sig = O.karras_sigmas(20)
        for i, st in enumerate(sched.steps):
            s = sig[i] * torch.ones(3)
            tm = O.times_from_sigma(s, False)
            assert st.n_inner == O.inner_steps_for(s, sig, tm.abt, n)
            assert all(torch.equal(a, b) for a, b in zip(st.times, tm))
            assert st.sigma == float(sig[i]) and st.sigma_next == float(sig[i + 1])
    assert [st.n_inner for st in HostSchedule(ks, 1, 5).steps] == [5] * 7 + [4, 4, 3, 3, 2, 1, 1] + [0] * 6
