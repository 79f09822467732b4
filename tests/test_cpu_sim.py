"""CPU checks of the simulated-archive path (pp_simulate_batch, WidebandPlan.simulate_batch, pplib.make_fake_pulsar):
the numpy restatement of its noise generator against the Random123 known answers, the uniform and Box-Muller
mapping, .par parsing, argument broadcasting and refusals, and the C struct layout against the ctypes binding."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import sim_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KAT = [  # Random123 kat_vectors: philox4x32 10 rounds, (ctr, key) -> out
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize("ctr,key,want", KAT, ids=["zeros", "ones", "pi"])
def test_philox_known_answers(ctr, key, want):
    got = sim_ref.philox4x32_10(ctr, key)
    assert [int(v) for v in got] == list(want)


def test_philox_is_elementwise():
    """the vectorised restatement gives each element what the scalar call gives"""
    c0 = np.array([0, 1, 2, 0xffffffff], dtype=np.uint64)
    got = sim_ref.philox4x32_10((c0, 7, 9, 11), (5, 6))
    for i, c in enumerate(c0):
        one = sim_ref.philox4x32_10((int(c), 7, 9, 11), (5, 6))
        assert [int(g[i]) for g in got] == [int(v) for v in one]


def test_uniform_mapping():
    x = np.array([0, 0xff, 0x100, 0x7fffffff, 0x80000000, 0xfffffeff, 0xffffffff], dtype=np.uint32)
    u = sim_ref.uniform(x)
    assert u.dtype == np.float32
    m = (x >> 8).astype(np.float64)
    exact = (m + 0.5) * 2.0 ** -24
    lower = exact < 0.5
    assert np.array_equal(u[lower].astype(np.float64), exact[lower])       # exact below 1/2
    assert np.all(np.abs(u.astype(np.float64) - exact) <= 2.0 ** -25)      # rounded to nearest above
    assert u[0] == np.float32(2.0 ** -25) and u[1] == u[0]                # the low byte is dropped
    assert u[-1] == np.float32(1.0)                                       # ties to even: the top value is 1
    assert np.all(np.diff(u.astype(np.float64)) >= 0)
    # the largest |z|: u0 = 2^-25
    rmax = np.sqrt(-2.0 * np.log(2.0 ** -25))
    assert 5.88 < rmax <= 5.9
    z0, z1, r = sim_ref.box_muller(np.array([0, 0xffffffff], dtype=np.uint32), np.array([0, 0x40000000], dtype=np.uint32))
    assert r[0] == pytest.approx(rmax, rel=1e-15) and r[1] == 0.0
    assert z0[0] == pytest.approx(rmax * np.cos(2 * np.pi * 2.0 ** -25), rel=1e-15)


def test_noise_layout_and_moments():
    """bins 4q..4q+3 of channel n of subint s come from counter (q, n, s lo, s hi); partial last quad"""
    z, r = sim_ref.noise(123, [0, 5, 2 ** 32 + 1], 3, 10)
    assert z.shape == (3, 3, 10) and r.shape == z.shape
    x = sim_ref.philox4x32_10((2, 1, 1, 1), (123, 0))                     # subint 2^32 + 1, channel 1, quad 2
    z0, z1, _ = sim_ref.box_muller(x[0], x[1])
    assert z[2, 1, 8] == z0 and z[2, 1, 9] == z1
    assert np.all(np.abs(z) <= 5.9)
    big, _ = sim_ref.noise(7, np.arange(8), 16, 4096)
    n = big.size
    assert abs(big.mean()) < 5 / np.sqrt(n) and abs(big.var() - 1) < 5 * np.sqrt(2.0 / n)


def test_read_ephemeris(tmp_path):
    from pulseportraiture_b200 import pplib
    par = tmp_path / "fake.par"
    par.write_text("PSRJ           J1234-5678\nF0             345.67890123456789  1\nF1  -1.5D-15 1\n"
                   "PEPOCH         55500\nDM             12.5\nRAJ 12:34:00\n")
    F0, F1, PEPOCH, DM, src = pplib.read_ephemeris(str(par))
    assert (F0, F1, PEPOCH, DM, src) == (345.67890123456789, -1.5e-15, 55500.0, 12.5, "J1234-5678")
    assert pplib.read_ephemeris(0.004) == (250.0, 0.0, 0.0, 0.0, "fake")
    with pytest.raises(ValueError):
        pplib.read_ephemeris(-1.0)
    bad = tmp_path / "bad.par"
    bad.write_text("PSRJ J0000+0000\nDM 3\n")
    with pytest.raises(ValueError):
        pplib.read_ephemeris(str(bad))


def test_make_fake_pulsar_broadcasting_and_refusals():
    from pulseportraiture_b200 import pplib
    assert np.array_equal(pplib._per_subint(0.25, 3, "phase"), [0.25] * 3)
    assert pplib._per_chan([1.0, 2.0], 3, 2, "scales").shape == (3, 2)
    assert pplib._per_chan(np.ones((3, 2)), 3, 2, "scales").shape == (3, 2)
    with pytest.raises(ValueError):
        pplib._per_subint([0.1, 0.2], 3, "phase")
    with pytest.raises(ValueError):
        pplib._per_chan(np.ones((2, 2)), 3, 2, "noise_stds")
    model = np.zeros((4, 64))
    with pytest.raises(ValueError):
        pplib.make_fake_pulsar(model, 0.004, npol=4, nchan=4, nbin=64)
    with pytest.raises(NotImplementedError):
        pplib.make_fake_pulsar(model, 0.004, scint=True, nchan=4, nbin=64)
    with pytest.raises(ValueError):
        pplib.make_fake_pulsar(model, 0.004, nsub=3, phase=[0.1, 0.2], nchan=4, nbin=64)
    with pytest.raises(ValueError):
        pplib.make_fake_pulsar(model, 0.004, nsub=3, noise_stds=-np.ones(4), nchan=4, nbin=64)


def test_sim_struct_layouts_match_the_header(tmp_path):
    from pulseportraiture_b200 import _ffi
    fields = [f for f, _ in _ffi.SimArgs._fields_]
    src = tmp_path / "layout.c"
    body = "".join('printf("%%zu ", offsetof(pp_sim_args_t, %s));' % f for f in fields)
    body += "".join('printf("%%zu ", offsetof(pp_sim_out_t, %s));' % f for f, _ in _ffi.SimOut._fields_)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ppb200.h"\nint main(void){%s'
                   'printf("%%zu %%zu\\n", sizeof(pp_sim_args_t), sizeof(pp_sim_out_t));return 0;}\n' % body)
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    want = [getattr(_ffi.SimArgs, f).offset for f in fields] + \
        [getattr(_ffi.SimOut, f).offset for f, _ in _ffi.SimOut._fields_] + \
        [C.sizeof(_ffi.SimArgs), C.sizeof(_ffi.SimOut)]
    assert got == want
