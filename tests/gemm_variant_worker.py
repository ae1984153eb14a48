"""Runs cases of test_gpu_gemm_variants.py in a process of its own, for the GEMM tuning knobs (XVB_GEMM_CTA, _WIDE, _BN,
_STORE, _BOX64) that the library reads once per process.  Not collected by pytest (no test_ prefix):

    XVB_GEMM_CTA=1 python tests/gemm_variant_worker.py --out result.json n256_production n128_pairs_f32 ...

Writes {case name: result} as JSON to --out -- the observed instantiation, the largest error/bound ratio, the failed
sentinel / mask / repeat checks and a digest of the output bits -- and prints the same as one line."""
import argparse
import json
import os
import sys
import traceback

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import test_gpu_gemm_variants as gv  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("cases", nargs="+")
    args = ap.parse_args()
    results = {}
    for name in args.cases:
        try:
            results[name] = gv.run_case(gv.CASES[name], sub_batch=False, expect_default=False)
        except Exception:
            results[name] = dict(name=name, observed=[], ratio=float("inf"), digest="",
                                 failures=[traceback.format_exc(limit=4)])
    with open(args.out, "w") as f:
        json.dump(results, f, indent=1)
    print(json.dumps({k: dict(observed=v["observed"], ratio=v["ratio"], failures=v["failures"]) for k, v in results.items()}))


if __name__ == "__main__":
    main()
