"""Record the diag_e digests of tests/metric_cases.py with a given build of the package.

    python tools/metric_digests.py [--pkg ep-stan_b200] [--out digests.json]

--pkg is the directory holding epstan/ and libepgpu.so (e.g. a checkout of an earlier commit, built with its
own build.py).  Prints one JSON object {case: {"digest": ..., "plan": {...}}}.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--pkg', default=os.path.join(ROOT, 'ep-stan_b200'))
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    sys.path[:0] = [os.path.abspath(args.pkg), ROOT, os.path.join(ROOT, 'tests')]
    from epstan import _lib
    import metric_cases
    res = {}
    for name in metric_cases.CASES:
        for k, (dg, plan) in metric_cases.run_case(_lib, name).items():
            res[k] = {'digest': dg, 'plan': plan}
    txt = json.dumps(res, indent=1, sort_keys=True)
    print(txt)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(txt)


if __name__ == '__main__':
    main()
