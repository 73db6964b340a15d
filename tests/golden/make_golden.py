"""Generates tests/golden/ctc_decoders.npz by running the REFERENCE's own numpy
decoders (the only part of the hot path that imports without TensorFlow):

    models/ctc/decoders/greedy_decoder.py:19-50      GreedyDecoder.__call__
    models/ctc/decoders/beam_search_decoder.py:53-152 BeamSearchDecoder.__call__

Run with a checkout of the reference repository:
    python tests/golden/make_golden.py <reference checkout>
The reference is called one utterance at a time, its canonical usage
(examples/librispeech/metrics/ctc.py:214-218).
"""
import os
import sys
import warnings

import numpy as np

sys.path.insert(0, sys.argv[1])
warnings.filterwarnings("ignore")
from models.ctc.decoders.beam_search_decoder import BeamSearchDecoder  # noqa: E402
from models.ctc.decoders.greedy_decoder import GreedyDecoder  # noqa: E402

CASES = [  # (T, C, beam, seed, peaky)
    (12, 4, 3, 0, 1.0), (30, 6, 5, 1, 2.0), (40, 29, 20, 2, 3.0), (60, 29, 20, 3, 6.0),
    (25, 10, 1, 4, 2.0), (50, 62, 10, 5, 4.0), (35, 5, 20, 6, 0.5), (80, 29, 20, 7, 8.0),
]


def main():
    out = {}
    for i, (T, C, beam, seed, peaky) in enumerate(CASES):
        rng = np.random.RandomState(seed)
        x = rng.randn(1, T, C) * peaky
        x[..., C - 1] += 0.5 * peaky          # blank-heavy like a trained CTC model
        p = np.exp(x - x.max(-1, keepdims=True))
        p /= p.sum(-1, keepdims=True)
        p = p.astype(np.float32)              # posteriors as sess.run would return them
        g = GreedyDecoder(blank_index=C - 1)(p, [T])
        b, s = BeamSearchDecoder(space_index=-1, blank_index=C - 1)(p, [T], beam_width=beam)
        out["probs_%d" % i] = p
        out["beam_%d" % i] = np.int32(beam)
        out["greedy_%d" % i] = np.asarray(g[0], dtype=np.int32)
        out["beam_labels_%d" % i] = np.asarray(b[0], dtype=np.int32)
        out["beam_score_%d" % i] = np.float64(s[0])
    out["n"] = np.int32(len(CASES))
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ctc_decoders.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main()
