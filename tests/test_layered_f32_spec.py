"""The binary32 layered min-sum specification (tests/layered_f32_oracle.c, DESIGN.md §3.7) on the CPU: value for value the fp64
specification orc_decode_layered where every binary32 operation is exact, and hand-worked single-check cases for signed zeros,
ties, the shortened-position LLR 99999.9 and the normalisation factor."""
import numpy as np
import pytest

import layered_f32_oracle as LF
from conftest import H_IRREGULAR


@pytest.fixture(scope="module")
def irregular():
    from oracle import oracle as O
    return O.Code(H_IRREGULAR)


def _integer_llrs(code, n, seed, mean):
    """Small integer LLRs (every sum the decoder forms stays far below 2^24: exact in binary32), with +-0 entries, 0 on the
    punctured and 1000 on the shortened positions, and one frame that does not converge."""
    rng = np.random.default_rng(seed)
    llr = np.clip(np.rint(rng.normal(mean, 6.0, (n, code.nc))), -20, 20)
    llr[0] = np.clip(np.rint(rng.normal(0.5, 8.0, code.nc)), -20, 20)
    llr[1, ::7] = -0.0
    llr[2, ::5] = 0.0
    llr[:, code.puncture] = 0.0
    llr[:, code.shorten] = 1000.0
    return llr


@pytest.mark.parametrize("which", ["h", "irregular"])
@pytest.mark.parametrize("iters, et", [(1, True), (5, False), (25, True), (50, True)])
def test_equals_fp64_specification_on_integer_llrs(oracle_code, irregular, which, iters, et):
    code = oracle_code if which == "h" else irregular
    layers = code.auto_layers()
    llr = _integer_llrs(code, 16, 31, 4.0 if which == "h" else 7.0)  # h.txt: rate 1/8 with 128 punctured; irregular: 0.43
    out, co, its = LF.decode(code, llr, layers, iters, et, f32=True)
    ro, rc, ri = code.decode_layered(llr, layers, iters, et, True)
    assert np.array_equal(its, ri) and np.array_equal(co, rc)
    assert np.array_equal(out.view(np.uint64), ro.view(np.uint64))          # -0.0 included
    assert np.abs(ro).max() < 2 ** 20
    # the batch loop's fp64 path is orc_decode_layered itself
    fo, fc, fi = LF.decode(code, llr, layers, iters, et, f32=False, threads=3)
    assert np.array_equal(fi, ri) and np.array_equal(fc, rc) and np.array_equal(fo.view(np.uint64), ro.view(np.uint64))
    if iters >= 25 and et:
        assert (ri < iters).any() and (ri == iters).any()                    # frames that converge and frames that fail


def _one_check(tmp_path, deg, shorten=()):
    """A code of one check on variables 0 .. deg-1 (one layer)."""
    from oracle import oracle as O
    p = tmp_path / ("check%d.txt" % deg)
    head = "shorten: %s\n" % " ".join(map(str, shorten)) if shorten else ""
    p.write_text(head + "".join("0 %d\n" % i for i in range(deg)))
    return O.Code(str(p))


def _bits(a):
    return np.asarray(a, dtype=np.float64).view(np.uint64).tolist()


@pytest.mark.parametrize("llr, scale, want", [
    # plain min-sum: c2v = sign product x minimum of the others; P = v2c + c2v
    ([3.0, -5.0, 7.0], 1.0, [-2.0, -2.0, 4.0]),
    # normalised by 48/64: c2v = [-3.75, 2.25, -2.25]
    ([3.0, -5.0, 7.0], 0.75, [-0.75, -2.75, 4.75]),
    # signed zeros: -0.0 is negative for the sign product; c2v = [-0.0, -0.0, +0.0], so -0.0 + -0.0 stays -0.0
    ([-0.0, -0.0, 3.0], 1.0, [-0.0, -0.0, 3.0]),
    # c2v = [-0.0, +0.0, -0.0]: x + (-x) rounds to +0.0
    ([0.0, -0.0, 2.0], 1.0, [0.0, 0.0, 2.0]),
    # ties: both smallest magnitudes are the minimum of the others for every edge; c2v = [-2, 2, -2, -2]
    ([2.0, -2.0, 2.0, 5.0], 1.0, [0.0, 0.0, 0.0, 3.0]),
    ([2.0, -2.0, 2.0, 5.0], 0.75, [0.5, -0.5, 0.5, 3.5]),
])
def test_single_check_by_hand(tmp_path, llr, scale, want):
    code = _one_check(tmp_path, len(llr))
    x = np.array([llr])
    for f32 in (True, False):                                                 # every operation here is exact in both
        out, co, its = LF.decode(code, x, code.auto_layers(), 1, False, f32=f32, ms_scale=scale)
        assert _bits(out[0]) == _bits(want) and its[0] == 1
        assert co[0].tolist() == [int(v <= 0) for v in want]


def test_shortened_position_llr_is_rounded_to_binary32(tmp_path):
    """99999.9 is 99999.8984375 in binary32; the posterior after c2v = -0.5 is 99999.3984375 (exact at that magnitude, whose
    binary32 spacing is 2^-7), where fp64 gives 99999.4.  The decisions are all zero: the frame stops after its first iteration."""
    code = _one_check(tmp_path, 3, shorten=(2,))
    assert code.n_short == 1 and code.nct == 2
    x = np.array([[1.5, -0.5, 99999.9]])
    out, co, its = LF.decode(code, x, code.auto_layers(), 10, True, f32=True)
    assert float(np.float32(99999.9)) == 99999.8984375
    assert _bits(out[0]) == _bits([1.0, 1.0, 99999.3984375]) and its[0] == 0 and co[0].tolist() == [0, 0, 0]
    ro, _, ri = code.decode_layered(x, code.auto_layers(), 10, True, True)
    assert ro[0].tolist() == [1.0, 1.0, 99999.9 - 0.5] and ri[0] == 0
    # without early termination the check keeps giving the same messages: the posteriors do not move
    out, _, its = LF.decode(code, x, code.auto_layers(), 3, False, f32=True)
    assert _bits(out[0]) == _bits([1.0, 1.0, 99999.3984375]) and its[0] == 3


def test_binary32_rounding_of_channel_llrs(oracle_code):
    """On non-integer LLRs the specification is the decoder on the binary32 values, not the fp64 one: decoding the LLRs
    already rounded to binary32 gives the same result bit for bit, and the fp64 specification differs."""
    _, llr = oracle_code.channel_frames("AWGN", -4.4, 3, 0, 0, 6)
    layers = oracle_code.auto_layers()
    a = LF.decode(oracle_code, llr, layers, 25, True, f32=True, ms_scale=0.75)
    b = LF.decode(oracle_code, llr.astype(np.float32).astype(np.float64), layers, 25, True, f32=True, ms_scale=0.75)
    assert all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(a, b))
    assert np.all(a[0].astype(np.float32).astype(np.float64) == a[0])           # posteriors are binary32 values
    ro, _, _ = oracle_code.decode_layered(llr, layers, 25, True, True, ms_scale=0.75)
    assert not np.array_equal(ro, a[0])


def test_sum_product_has_no_binary32_specification(oracle_code):
    with pytest.raises(ValueError, match="no exact specification"):
        LF.decode(oracle_code, np.zeros((1, oracle_code.nc)), oracle_code.auto_layers(), 5, True, f32=True, minsum=False)
