"""
Generates tests/golden/oracle_snapshot.npz: the ORACLE's own outputs (oracle/sygnals_oracle.py, not the reference
package) on the seeded inputs of tests/test_oracle_vs_reference.py.  The snapshot tests there are a regression guard:
they catch any change of the oracle's results.  They do not show that the oracle matches the reference; only the live
tests of that module do, where the reference package is installed.  This file was written from the oracle as it stood
when the snapshot tests were added, on a machine without the reference package.  Regenerate it only for an intended
change of the oracle's results, and preferably where the live tests run and pass:

    python tests/golden/make_oracle_snapshot.py

Stored per case: extract_features' full output (column names in order + float64 rows); for compute_stft the shape, a
float64 checksum of the whole transform and a fixed seeded sample of 1024 bins; for segment_fixed_length the count, the
lengths and a checksum of every segment; format_feature_vectors_per_segment's full output.
"""
import logging
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_oracle_vs_reference as T  # noqa: E402
from oracle import sygnals_oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_snapshot.npz")


def main():
    warnings.simplefilter("ignore")
    logging.disable(logging.CRITICAL)
    d = {}
    for i, case in enumerate(T.EF_CASES):
        y, sr, fl, hop = T.ef_input(*case)
        r = O.extract_features(y, sr, T.FEATS, frame_length=fl, hop_length=hop, feature_params=T.EF_PARAMS)
        d[f"ef{i}_names"] = np.array(list(r))
        d[f"ef{i}_rows"] = np.stack([r[k] for k in r])
    y = T.seg_input()
    for i, kw in enumerate(T.SEG_CASES):
        segs = O.segment_fixed_length(y, 1000, **kw)
        d[f"seg{i}_lengths"] = np.array([len(s) for s in segs], dtype=np.int64)
        d[f"seg{i}_checksums"] = np.array([T.checksum(s) for s in segs]).reshape(len(segs), 3)
    for i, kw in enumerate(T.STFT_CASES):
        D = O.compute_stft(y, **kw)
        d[f"stft{i}_shape"] = np.array(D.shape, dtype=np.int64)
        d[f"stft{i}_checksum"] = T.checksum(np.abs(D))
        d[f"stft{i}_sample"] = D.ravel()[T.stft_sample_index(D.size)]
    feats, segs = T.agg_input()
    for i, agg in enumerate(T.AGG_CASES):
        d[f"agg{i}"] = O.format_feature_vectors_per_segment(feats, segs, agg)
    np.savez_compressed(OUT, **d)
    print(OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
