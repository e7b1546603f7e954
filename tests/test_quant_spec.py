"""The fixed-point layered min-sum specification (tests/quant_oracle.c, DESIGN.md §3.7) on the CPU: the quantiser and the check
rule on hand-worked values, the equivalence with the fp64 layered min-sum (orc_decode_layered) on integer LLRs, and the CLI's
parse-time errors for --quantize."""
import os
import subprocess

import numpy as np
import pytest

import quant_oracle as Q
from conftest import H_FILE, ROOT

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")


def test_quantizer_rounds_half_away_and_clamps():
    q = Q.quant(6, 6, 8, 0.5)                                   # M(6) = 31
    vals = [0.0, -0.0, 0.25, -0.25, 0.2499, 0.75, -0.75, 1.0, -1.2, 15.25, 15.5, -15.5, 16.0, 99999.9, -99999.9, 1e300]
    want = [0, 0, 1, -1, 0, 2, -2, 2, -2, 31, 31, -31, 31, 31, -31, 31]
    assert Q.quantize(vals, q).tolist() == want
    q = Q.quant(4, 4, 6, 1.0)                                   # M(4) = 7
    assert Q.quantize([0.5, -0.5, 1.5, 2.5, -2.5, 6.5, 7.4, 7.6, -8.0, 99999.9], q).tolist() == [1, -1, 2, 3, -3, 7, 7, 7, -7, 7]
    # the division is correctly rounded in fp64 before the rounding: 0.3 / 0.1 = 2.9999999999999996 -> 3, 0.15 / 0.1 = 1.4999999999999998 -> 1
    q = Q.quant(8, 8, 8, 0.1)
    assert Q.quantize([0.3, 0.15, -0.15, 0.25], q).tolist() == [3, 1, -1, 3]


@pytest.mark.parametrize("v, params, want", [
    # plain min-sum: min of the others, sign product of the others (0 counts as positive)
    ([3, -5, 7], (8, 8, 8, 0, 8), [-5, 3, -3]),
    ([0, -2, 4], (8, 8, 8, 0, 8), [-2, 0, 0]),
    ([0, 0, -1], (8, 8, 8, 0, 8), [0, 0, 0]),
    ([-4, -6], (8, 8, 8, 0, 8), [-6, -4]),
    # message clip: magnitudes above M(Qm) = 7 count as 7
    ([100, -90, 120], (8, 4, 8, 0, 8), [-7, 7, -7]),
    ([100, -3, 120], (8, 4, 8, 0, 8), [-3, 7, -3]),
    # offset: max(m - beta, 0), offset to zero keeps the sign rule harmless
    ([3, -5, 7], (8, 8, 8, 2, 8), [-3, 1, -1]),
    ([1, -2, 9], (8, 8, 8, 2, 8), [0, 0, 0]),
    # normalisation a/8, floor before the offset: floor(5 * 6 / 8) = 3, floor(3 * 6 / 8) = 2
    ([3, -5, 7], (8, 8, 8, 0, 6), [-3, 2, -2]),
    ([3, -5, 7], (8, 8, 8, 1, 6), [-2, 1, -1]),
    ([31, 31, -31, 31], (6, 6, 6, 0, 1), [-3, -3, 3, -3]),
])
def test_check_rule_by_hand(v, params, want):
    ch, msg, post, beta, a = params
    assert Q.check(v, Q.quant(ch, msg, post, 1.0, beta, a)).tolist() == want


def test_layered_update_saturates_the_posterior(oracle_code):
    """With 4-bit posteriors every posterior stays in [-7, 7], and the output is P * step."""
    q = Q.quant(4, 4, 4, 0.25)
    rng = np.random.default_rng(3)
    llr = rng.normal(1.0, 2.0, (4, oracle_code.nc))
    out, co, its, post, clips = Q.decode(oracle_code, llr, oracle_code.auto_layers(), q, 10, False)
    assert np.abs(post).max() == 7 and clips > 0
    assert np.array_equal(out, post * 0.25) and np.array_equal(co, (post <= 0).astype(np.uint8))


def _integer_llrs(nc, n, seed):
    rng = np.random.default_rng(seed)
    base = np.clip(np.rint(rng.normal(3.0, 6.0, (n, nc))), -20, 20)
    base[0] = np.clip(np.rint(rng.normal(0.5, 8.0, nc)), -20, 20)   # a frame that does not converge
    return base


@pytest.fixture(scope="module")
def bg1():
    from conftest import large_code_files
    from oracle import oracle as O
    return O.Code(large_code_files()["bg1"])


@pytest.mark.parametrize("which", ["h", "bg1"])
@pytest.mark.parametrize("iters, et", [(1, True), (5, False), (20, True), (20, False), (50, True)])
def test_equals_fp64_layered_min_sum_on_integer_llrs(oracle_code, bg1, which, iters, et):
    """Qp = Qm = 16, a = 8, beta = 0 and integer multiples of the step below 2^15 steps: the integer decoder is the fp64 layered
    min-sum, value for value (no saturation or clip ever changed a value, so no fp64 value reached 2^15 steps)."""
    code = oracle_code if which == "h" else bg1
    layers = code.auto_layers()
    n = 12 if which == "h" else 3
    for step in (1.0, 0.5):
        llr = _integer_llrs(code.nc, n, 11 + iters) * step
        q = Q.quant(16, 16, 16, step)
        out, co, its, post, clips = Q.decode(code, llr, layers, q, iters, et)
        ro, rc, ri = code.decode_layered(llr, layers, iters, et, True)
        assert clips == 0 and np.abs(ro).max() < 2 ** 15 * step
        assert np.array_equal(its, ri) and np.array_equal(co, rc)
        assert np.array_equal(out, ro)                                   # values: -0.0 == 0.0
        assert np.array_equal(post * step, ro)
        if which == "h" and iters >= 20 and et:
            assert (ri < iters).any() and (ri == iters).any()            # frames that converge and frames that fail


def _cli(tmp_path, *extra):
    out = tmp_path / "o.txt"
    r = subprocess.run([CLI, H_FILE, str(out), "0", "2", "1", *extra], capture_output=True, text=True)
    return r, out


LAYERED_MS = ("--schedule", "layered", "--decoding", "BP_MS")


@pytest.mark.parametrize("extra, message", [
    (("--quantize", "6,6,8", "--llr-step", "0.5", "--decoding", "BP_MS"), "--quantize needs --schedule layered"),
    (("--quantize", "6,6,8", "--llr-step", "0.5", "--schedule", "layered"), "--quantize needs --decoding BP_MS"),
    (("--quantize", "6,6,8", "--llr-step", "0.5", "--channel", "BEC") + LAYERED_MS, "--quantize does not apply to --channel BEC"),
    (("--quantize", "6,6,8", "--llr-step", "0.5", "--modulation", "4") + LAYERED_MS, "--quantize needs --modulation 2"),
    (("--quantize", "6,6,8") + LAYERED_MS, "--quantize needs --llr-step"),
    (("--quantize", "6,6,8", "--llr-step", "0") + LAYERED_MS, "--llr-step must be > 0"),
    (("--llr-step", "0.5",) + LAYERED_MS, "--llr-step applies to --quantize only"),
    (("--ms-offset", "1",) + LAYERED_MS, "--ms-offset applies to --quantize only"),
    (("--quantize", "6,6", "--llr-step", "0.5") + LAYERED_MS, "--quantize expects CH,MSG,POST"),
    (("--quantize", "6,8,7", "--llr-step", "0.5") + LAYERED_MS, "bit widths"),
    (("--quantize", "9,6,8", "--llr-step", "0.5") + LAYERED_MS, "bit widths"),
    (("--quantize", "1,1,8", "--llr-step", "0.5") + LAYERED_MS, "bit widths"),
    (("--quantize", "6,6,17", "--llr-step", "0.5") + LAYERED_MS, "bit widths"),
    (("--quantize", "6,3,8", "--llr-step", "0.5", "--ms-offset", "3") + LAYERED_MS, "--ms-offset must be"),
    (("--quantize", "6,6,8", "--llr-step", "0.5", "--ms-offset", "-1") + LAYERED_MS, "--ms-offset must be"),
    (("--quantize", "6,6,8", "--llr-step", "0.5", "--ms-scale", "0.8") + LAYERED_MS, "--ms-scale must be a multiple of 1/8"),
])
def test_cli_rejects_bad_quantize_arguments(built_lib, tmp_path, extra, message):
    r, out = _cli(tmp_path, *extra)
    assert r.returncode != 0 and message in r.stdout, r.stdout
    assert not out.exists()


def test_cli_documents_quantize(built_lib):
    r = subprocess.run([CLI, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and all(f in r.stdout for f in ("--quantize", "--llr-step", "--ms-offset"))
