"""Generates tests/golden/input_pipeline.npz by running the REFERENCE's own numpy input
transforms (they import without TensorFlow):

    utils/io/inputs/frame_stacking.py:14-85   stack_frame
    utils/io/inputs/splicing.py:9-73          do_splice

and, on the way, asserts that the closed-form restatement in oracle/inputs.py reproduces them
bit for bit on a wider random sweep.  Run with a checkout of the reference repository:
    python tests/golden/make_golden_inputs.py <reference checkout>
"""
import os
import sys

import numpy as np

sys.path.insert(0, sys.argv[1])
from utils.io.inputs.frame_stacking import stack_frame  # noqa: E402
from utils.io.inputs.splicing import do_splice  # noqa: E402

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from oracle import inputs as oin  # noqa: E402

CASES = [  # (T, num_channels, num_stack, num_skip, splice, seed)
    (17, 4, 1, 1, 1, 0), (17, 4, 3, 3, 1, 1), (20, 5, 3, 2, 1, 2), (9, 2, 2, 1, 5, 3),
    (31, 3, 1, 1, 11, 4), (26, 4, 2, 2, 11, 5), (5, 2, 3, 3, 3, 6), (40, 8, 3, 3, 1, 7),
]


def ref_pipeline(x, S, K, P):
    st = stack_frame([x], S, K)[0] if S > 1 else x
    st = np.asarray(st)
    sp = do_splice(st[None].astype(np.float64), splice=P, batch_size=1, num_stack=S)[0]
    return st, sp


def main():
    # wide sweep: closed form == reference
    rng = np.random.RandomState(123)
    n = 0
    for T in (1, 2, 3, 7, 16, 33):
        for nch in (1, 3):
            for S, K in ((1, 1), (2, 1), (2, 2), (3, 2), (3, 3), (4, 3)):
                for P in (1, 3, 5, 11):
                    x = rng.randn(T, nch * 3).astype(np.float32)
                    st, sp = ref_pipeline(x, S, K, P)
                    st2 = oin.stack_frame(x, S, K)
                    assert st2.shape == st.shape and np.array_equal(st2, st), (T, nch, S, K)
                    sp2 = oin.do_splice(st2, P, S)
                    assert sp2.shape == sp.shape and np.array_equal(sp2.astype(np.float64), sp), (T, nch, S, K, P)
                    n += 1
    print("closed form == reference on %d configurations" % n)
    out = {}
    for i, (T, nch, S, K, P, seed) in enumerate(CASES):
        x = np.random.RandomState(seed).randn(T, nch * 3).astype(np.float32)
        st, sp = ref_pipeline(x, S, K, P)
        out["x_%d" % i] = x
        out["stacked_%d" % i] = np.asarray(st, np.float32)
        out["spliced_%d" % i] = np.asarray(sp, np.float32)
        out["cfg_%d" % i] = np.array([T, nch, S, K, P], np.int64)
    out["n_cases"] = np.array(len(CASES))
    path = os.path.join(os.path.dirname(__file__), "input_pipeline.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main()
