"""The RAYLEIGH channel's specification (tests/rayleigh_oracle.c, DESIGN.md §3.2) on the CPU: the distribution and block
structure of the fading coefficients, the faded LLRs against the formula rebuilt from the AWGN noise, and the CLI's argument
checks, which run before any device is touched."""
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import rayleigh_oracle as R
from conftest import H_FILE, ROOT

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")
SEED, POINT = 0x1234_5678_9ABC, 3


def test_coefficients_are_rayleigh_with_unit_power():
    # 2^17 coefficients: 8 frames x 16384 indices (two of the frames above 2^32)
    h = np.concatenate([R.coeffs(SEED, POINT, f, range(16384)) for f in (0, 1, 2, 7, 1000, 123456, (1 << 32) + 5, (1 << 40) + 1)])
    assert h.size >= 1 << 16 and np.all(h > 0)
    assert abs(np.mean(h * h) - 1.0) < 0.01
    ks = stats.kstest(h, lambda v: 1.0 - np.exp(-v * v))
    assert ks.pvalue > 0.01, ks


def test_coefficients_are_independent_across_indices_and_frames():
    h = R.coeffs(SEED, POINT, 9, range(1 << 15))
    r = np.corrcoef(h[:-1], h[1:])[0, 1]
    assert abs(r) < 4 / math.sqrt(h.size), r
    h0 = np.array([R.coeffs(SEED, POINT, f, [0])[0] for f in range(4096)])   # coefficient 0 of consecutive frames (L = 0)
    r = np.corrcoef(h0[:-1], h0[1:])[0, 1]
    assert abs(r) < 4 / math.sqrt(h0.size), r
    other = R.coeffs(SEED, POINT + 1, 9, range(4096))                        # another sweep point
    assert abs(np.corrcoef(h[:4096], other)[0, 1]) < 4 / math.sqrt(4096)


@pytest.mark.parametrize("L", [1, 7, 0])
def test_coefficients_constant_within_blocks_of_L(oracle_code, L):
    # at 160 dB the noise is negligible: LLR / (2 / sigma^2) = (z sigma + h) h = h^2 (1 + O(1e-8 / h)) reveals every h
    x = 160.0
    scale = 2.0 / math.pow(10, -x / 10)
    t = np.arange(oracle_code.nct)
    c = t // L if L else np.zeros_like(t)
    for frame in (5, 6):
        _, llr = R.channel_frames(oracle_code, x, L, SEED, POINT, frame, 1)
        h = np.sqrt(llr[0][oracle_code.bit_pos] / scale)
        want = R.coeffs(SEED, POINT, frame, range(int(c[-1]) + 1))
        assert np.unique(want).size == want.size
        assert np.allclose(h, want[c], rtol=1e-4, atol=0)
        if L != 1:
            assert all(np.ptp(h[c == j]) < 1e-4 * want[j] for j in range(want.size))


@pytest.mark.parametrize("L", [1, 7, 0])
@pytest.mark.parametrize("with_gen", [False, True])
def test_faded_llrs_equal_the_formula(oracle_code, oracle_gen, L, with_gen):
    from oracle import oracle as O
    gen = oracle_gen if with_gen else None
    x, frame0, n = 1.5, (1 << 32) + 17, 3
    cw, llr = R.channel_frames(oracle_code, x, L, SEED, POINT, frame0, n, gen=gen)
    cw_awgn, llr_awgn = oracle_code.channel_frames("AWGN", x, SEED, POINT, frame0, n, gen=gen)
    assert np.array_equal(cw, cw_awgn)
    if with_gen:
        assert cw.any()
    sigma2 = math.pow(10, -x / 10)
    sigma, scale = math.sqrt(sigma2), 2.0 / sigma2
    nb = (oracle_code.nct + 3) // 4
    want = llr_awgn.copy()   # punctured 0.0 and shortened 99999.9 as for AWGN
    for f in range(n):
        for t in range(oracle_code.nct):
            q, k = t % nb, t // nb
            z = O.normal_block(SEED, POINT, frame0 + f, q)[k]
            h = R.coeffs(SEED, POINT, frame0 + f, [t // L if L else 0])[0]
            v = oracle_code.bit_pos[t]
            y = z * sigma + (-h if cw[f, v] else h)
            want[f, v] = (y * h) * scale
    assert np.array_equal(llr.view(np.uint64), want.view(np.uint64))


def _cli(tmp_path, *extra):
    out = tmp_path / "o.txt"
    r = subprocess.run([CLI, H_FILE, str(out), "0", "2", "1", *extra], capture_output=True, text=True)
    return r, out


@pytest.mark.parametrize("extra, message", [
    (("--channel", "RAYLEIGH", "--coherence", "-1"), "--coherence must be >= 0"),
    (("--coherence", "4"), "--coherence applies to --channel RAYLEIGH only"),
    (("--channel", "AWGN", "--coherence", "1"), "--coherence applies to --channel RAYLEIGH only"),
    (("--channel", "RAYLEIGH", "--modulation", "4"), "--channel RAYLEIGH is BPSK only"),
])
def test_cli_rejects_bad_fading_arguments(built_lib, tmp_path, extra, message):
    r, out = _cli(tmp_path, *extra)
    assert r.returncode != 0 and message in r.stdout, r.stdout
    assert not out.exists()


def test_cli_documents_the_channel(built_lib):
    r = subprocess.run([CLI, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "RAYLEIGH" in r.stdout and "--coherence" in r.stdout
