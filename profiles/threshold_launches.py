"""Kernel launches (`ctx.launches`, bq_launch_count) of each thresholding entry point on a `synth.cv_tables` cohort:
`apply`, `detect`, `from_cv`, and `FoldSet.from_cv` called twice as the nested-CV caller does (tile threshold first,
then the slide thresholds with it fixed).  Two builds that do the same device work print the same JSON line.

    python profiles/threshold_launches.py
"""
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
warnings.simplefilter("ignore")


def main():
    from biscuit_b200 import _ffi, threshold
    from oracle import synth

    ctx = _ffi.default_context()
    folds = synth.cv_tables(k=4, n_slides=40, tiles_per_slide=500, seed0=11)
    out = {}

    def count(name, fn):
        before = ctx.launches
        result = fn()
        out[name] = ctx.launches - before
        return result

    th = count("from_cv", lambda: threshold.from_cv([f.copy() for f in folds]))
    count("detect", lambda: threshold.detect(folds[0].copy()))
    count("apply", lambda: threshold.apply(folds[1].copy(), **th))
    with threshold.FoldSet([f.copy() for f in folds]) as fs:
        first = count("FoldSet.from_cv#1", lambda: fs.from_cv(tile_uq="detect", slide_uq=None))
        count("FoldSet.from_cv#2", lambda: fs.from_cv(tile_uq=first["tile_uq"], slide_uq="detect"))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
