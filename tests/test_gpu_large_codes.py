"""GPU parity on the two large BASELINE configs (3: NR-BG1-shaped QC code Z=384, 4: DVB-S2-shaped IRA code
n=64800; codes/gen_codes.py explains why they are structure-matched rather than standard-exact): global
(HBM/L2) residency, check degrees up to 19, variable degrees up to 30.  Same bars as test_gpu_parity.py.

The comparand is the UNMODIFIED reference decoder: its outputs on these very frames are stored in
tests/golden/large_codes_ref.npz (tests/golden/make_large_golden.py), and the C oracle, which supplies the full arrays, is
checked against that record on every call (it is also the frame generator: the counter-based channel specification)."""
import numpy as np
import pytest

from conftest import large_code_files, reference_outputs

pytestmark = pytest.mark.gpu

BP_RTOL = 1e-4  # tolerance stated by BASELINE.json north_star for BP posterior LLRs

CASES = {"bg1": dict(conv=0.0, hard=-1.0), "dvbs2": dict(conv=2.0, hard=0.5)}


@pytest.fixture(scope="module", params=["bg1", "dvbs2"])
def big(request, built_lib):
    from libldpc_b200 import api
    from oracle import oracle as O
    path = large_code_files()[request.param]
    ctx = api.Context(path, "", device=0)
    yield request.param, ctx, O.Code(path), path
    ctx.close()


def _rel_err(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-9)


def test_sizes(big):
    name, ctx, oc, path = big
    want = {"bg1": (26112, 17664, 121344, 25344), "dvbs2": (64800, 32400, 226799, 64800)}[name]
    assert (ctx.nc, ctx.mc, ctx.nnz, ctx.nct) == want == (oc.nc, oc.mc, oc.nnz, oc.nct)


@pytest.mark.parametrize("prec_fpc", [(0, 0), (0, 8)])
def test_minsum_bit_exact(big, prec_fpc):
    from libldpc_b200 import api
    name, ctx, oc, path = big
    ctx.set_tuning(precision=api.F64, residency=api.AUTO, frames_per_cta=prec_fpc[1])
    for x, et, iters in ((CASES[name]["conv"], True, 50), (CASES[name]["hard"], True, 12), (CASES[name]["conv"], False, 6)):
        cw, llr = oc.channel_frames("AWGN", x, 3, 1, 0, 7)
        ro, rc, ri = reference_outputs(name, path, oc, llr, "BP_MS", iters, et)
        out, hard, its = ctx.decode_batch(llr, "BP_MS", iters, et)
        assert np.array_equal(its, ri), (name, x)
        assert np.array_equal(hard, rc), (name, x)
        assert np.array_equal(out.view(np.uint64), ro.view(np.uint64)), (name, x)
    ctx.set_tuning(frames_per_cta=0)


def test_bp_within_tolerance(big):
    from libldpc_b200 import api
    name, ctx, oc, path = big
    ctx.set_tuning(precision=api.F64, residency=api.AUTO, frames_per_cta=0)
    for x, et, iters in ((CASES[name]["conv"] + 0.5, True, 50), (CASES[name]["hard"], False, 2), (CASES[name]["hard"], False, 50)):
        cw, llr = oc.channel_frames("AWGN", x, 4, 0, 0, 3 if iters == 50 and not et else 5)
        ro, rc, ri = reference_outputs(name, path, oc, llr, "BP", iters, et)
        out, hard, its = ctx.decode_batch(llr, "BP", iters, et)
        assert np.array_equal(its, ri), (name, x)
        assert (hard == rc).mean() >= 0.9999
        assert _rel_err(out, ro).max() < BP_RTOL


def test_fused_sim_counters_match_oracle_on_dumped_llrs(big):
    """channel -> decode -> accounting fused on the GPU == the oracle decoding the LLRs the GPU channel dumps."""
    name, ctx, oc, path = big
    n, x = 24, CASES[name]["conv"] - 0.4
    g = ctx.sim_point("AWGN", x, seed=2, point=1, frame0=10, nframes=n, decoding="BP_MS", iterations=30, early_term=True)
    cw, llr = ctx.channel("AWGN", x, seed=2, point=1, frame0=10, n=n)
    out, co, its = oc.decode(llr, 30, True, True)
    errs = (co[:, oc.bit_pos] != 0).sum(1)
    assert g["frames"] == n and g["iters"] == int(its.sum())
    assert g["fec"] == int((errs > 0).sum()) and g["bec"] == int(errs.sum())
    if len(oc.puncture):
        assert np.all(llr[:, oc.puncture] == 0.0)


def test_bsc_two_valued_llrs_bit_exact(big):
    """BSC-style inputs (LLR in {+-delta, 0}: exact ties and exact zeros everywhere) against the reference decoder."""
    from libldpc_b200 import api
    name, ctx, oc, path = big
    ctx.set_tuning(precision=api.F64, residency=api.AUTO, frames_per_cta=0)
    eps = {"bg1": 0.09, "dvbs2": 0.06}[name]
    cw, llr = oc.channel_frames("BSC", eps, 6, 0, 0, 4)
    for et, iters in ((True, 50), (False, 5)):
        ro, rc, ri = reference_outputs(name, path, oc, llr, "BP_MS", iters, et)
        out, hard, its = ctx.decode_batch(llr, "BP_MS", iters, et)
        assert np.array_equal(its, ri) and np.array_equal(hard, rc)
        assert np.array_equal(out.view(np.uint64), ro.view(np.uint64))
