import functools
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H_FILE = os.path.join(ROOT, "codes", "ref_h_n1152_m1024.txt")
G_FILE = os.path.join(ROOT, "codes", "ref_g_k128_n1152.txt")
GOLDEN = os.path.join(ROOT, "tests", "golden")
H_IRREGULAR = os.path.join(GOLDEN, "irregular_h.txt")   # committed; written once by tests/golden/make_irregular_golden.py


def large_code_files():
    """BASELINE configs 3/4 code files, generated deterministically on first use (codes/gen_codes.py)."""
    sys.path.insert(0, os.path.join(ROOT, "codes"))
    import gen_codes
    return gen_codes.ensure()


LARGE_REF = os.path.join(GOLDEN, "large_codes_ref.npz")   # written by tests/golden/make_large_golden.py


def large_case_key(name, llr, decoding, iters, et):
    """Names one decode of the large codes by its inputs: code, decoder settings and a digest of the LLRs."""
    import hashlib
    import numpy as np
    digest = hashlib.sha256(np.ascontiguousarray(llr, dtype=np.float64).tobytes()).hexdigest()[:16]
    return "%s:%s:%d:%d:%s" % (name, decoding, iters, int(et), digest)


@functools.lru_cache(maxsize=None)
def _large_ref_cases():
    return _load_cases(LARGE_REF)


def reference_outputs(name, path, oc, llr, decoding, iters, et):
    """The reference decoder's outputs on the large codes: the oracle's full outputs, checked against what the unmodified
    reference decoder (its ldpc_decoder::decode through oracle/dump_ref.cpp) returned for the same inputs.  Stored per
    case: iteration counts, hard decisions, a SHA-256 of the posterior LLRs' bytes and a fixed sample of them."""
    import hashlib
    import numpy as np
    cases = _large_ref_cases()
    with open(path, "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == str(cases["code_" + name]["sha256"]), \
            "%s differs from the code file the reference outputs were recorded on (codes/gen_codes.py)" % path
    key = large_case_key(name, llr, decoding, iters, et)
    assert key in cases, "no stored reference outputs for %s: regenerate with tests/golden/make_large_golden.py" % key
    ref = cases[key]
    out, co, its = oc.decode(llr, iters, et, decoding == "BP_MS")
    assert np.array_equal(its, ref["iters"]), key
    assert np.array_equal(np.packbits(co, axis=1), ref["co_bits"]), key
    assert np.array_equal(out[:, ref["sample_idx"]].view(np.uint64), ref["llr_out_sample"].view(np.uint64)), key
    assert hashlib.sha256(out.tobytes()).hexdigest() == str(ref["llr_out_sha256"]), key
    return out, co, its


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


@pytest.fixture(scope="session")
def built_lib():
    """Builds (if stale) and loads libldpc_b200/libldpc.so; never falls back to anything else."""
    from libldpc_b200 import build as B
    B.build()
    from libldpc_b200 import api
    return api.load_library()


@pytest.fixture(scope="session")
def oracle_code():
    from oracle import oracle as O
    return O.Code(H_FILE)


@pytest.fixture(scope="session")
def oracle_gen():
    from oracle import oracle as O
    return O.Code(G_FILE, matrix_only=True)


@pytest.fixture(scope="session")
def golden_cases():
    import numpy as np
    z = np.load(os.path.join(GOLDEN, "decode_cases.npz"))
    cases = {}
    for key in z.files:
        name, field = key.split("/")
        cases.setdefault(name, {})[field] = z[key]
    return cases


def _load_cases(path):
    import numpy as np
    z = np.load(path)
    cases = {}
    for key in z.files:
        name, field = key.split("/")
        cases.setdefault(name, {})[field] = z[key]
    return cases


@pytest.fixture(scope="session")
def irregular_cases():
    """Outputs of the unmodified reference decoder (oracle/_ref/dump_ref decode) on the irregular code."""
    return _load_cases(os.path.join(GOLDEN, "irregular_cases.npz"))


@pytest.fixture(scope="session")
def gpu_ctx(built_lib):
    from libldpc_b200 import api
    if built_lib.ldpc_b200_device_count() < 1:
        pytest.fail("no CUDA device visible: GPU tests must run on the GPU box (there is no CPU fallback)")
    ctx = api.Context(H_FILE, G_FILE, device=0)
    yield ctx
    ctx.close()
