"""Records the UNMODIFIED reference decoder's outputs on the two large codes (BASELINE configs 3/4, codes/gen_codes.py).

  tests/golden/large_codes_ref.npz   per decode case (key: conftest.large_case_key — code, decoder settings, LLR digest):
                                     iters, co_bits (hard decisions, np.packbits along the frame), llr_out_sha256
                                     (SHA-256 of the float64 posteriors), sample_idx + llr_out_sample (a fixed sample of
                                     them); per code: code_<name>/sha256 of the generated code file

The inputs are the ones tests/test_gpu_large_codes.py and tests/test_oracle_golden.py decode: frames of the oracle's
counter-based channel.  The full posteriors of these codes do not fit a small file, so they are pinned by digest; the
tests take the full arrays from the C oracle after checking it against this record.

Usage:  python tests/golden/make_large_golden.py      (needs oracle/_ref/dump_ref, built by `make -C oracle` from the
        reference sources; about a minute)
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from conftest import LARGE_REF, large_case_key, large_code_files  # noqa: E402
from oracle import oracle as O  # noqa: E402

SAMPLE = 64          # posterior LLRs stored per frame


def cases(name):
    """(channel, x, seed, point, nframes, decoding, iterations, early_term) of every decode the tests run on `name`."""
    conv, hard = {"bg1": (0.0, -1.0), "dvbs2": (2.0, 0.5)}[name]
    out = []
    # test_gpu_large_codes.py: test_minsum_bit_exact, test_bp_within_tolerance, test_bsc_two_valued_llrs_bit_exact
    for x, et, it in ((conv, True, 50), (hard, True, 12), (conv, False, 6)):
        out.append(("AWGN", x, 3, 1, 7, "BP_MS", it, et))
    for x, et, it in ((conv + 0.5, True, 50), (hard, False, 2), (hard, False, 50)):
        out.append(("AWGN", x, 4, 0, 3 if it == 50 and not et else 5, "BP", it, et))
    eps = {"bg1": 0.09, "dvbs2": 0.06}[name]
    for et, it in ((True, 50), (False, 5)):
        out.append(("BSC", eps, 6, 0, 4, "BP_MS", it, et))
    # test_oracle_golden.py: test_oracle_equals_reference_on_large_codes
    x = {"bg1": -0.6, "dvbs2": 1.0}[name]
    for dec, it, et in (("BP_MS", 50, True), ("BP_MS", 4, False), ("BP", 3, False)):
        out.append(("AWGN", x, 11, 0, 2, dec, it, et))
    return out


def main():
    if not O.ref_available():
        raise SystemExit("oracle/_ref/dump_ref is missing: build it with `make -C oracle REF=<reference sources>`")
    store = {}
    tmp = tempfile.TemporaryDirectory()
    for name, path in large_code_files().items():
        with open(path, "rb") as f:
            store["code_%s/sha256" % name] = np.array(hashlib.sha256(f.read()).hexdigest())
        oc = O.Code(path)
        idx = np.sort(np.random.default_rng(oc.nc).choice(oc.nc, SAMPLE, replace=False)).astype(np.int32)
        for ch, x, seed, point, n, dec, it, et in cases(name):
            cw, llr = oc.channel_frames(ch, x, seed, point, 0, n)
            key = large_case_key(name, llr, dec, it, et)
            if key + "/iters" in store:
                continue
            r = O.ref_decode(path, dec, it, et, llr, tmp=os.path.join(tmp.name, "dec"))
            store[key + "/iters"] = r["iters"]
            store[key + "/co_bits"] = np.packbits(r["co"], axis=1)
            store[key + "/llr_out_sha256"] = np.array(hashlib.sha256(r["llr_out"].tobytes()).hexdigest())
            store[key + "/sample_idx"] = idx
            store[key + "/llr_out_sample"] = r["llr_out"][:, idx]
            print(key, "iters", r["iters"])
    np.savez_compressed(LARGE_REF, **store)
    print(LARGE_REF, os.path.getsize(LARGE_REF), "bytes")


if __name__ == "__main__":
    main()
