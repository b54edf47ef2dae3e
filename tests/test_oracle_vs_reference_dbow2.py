"""The oracle's DBoW2 restatement (oracle/bow_oracle.cpp) against the REFERENCE'S OWN DBoW2 code: oracle/_ref/libdbow2_ref.so is
cslam/thirdparty/DBoW2 compiled where it lies (oracle/Makefile `ref`, stand-in OpenCV header oracle/ref_stub/) — the one piece of the
hot path's neighbourhood that builds in this image.  Vocabulary text loader, word / node numbering, tree descent with its first-minimum
rule, FORB::distance, BowVector / FeatureVector arithmetic for every scoring and weighting type: exact, doubles bit for bit.
The reference's outputs are stored under tests/golden/reference (tests/reference_outputs.py)."""
import os
import tempfile

import numpy as np
import pytest

from ccm_slam_b200 import synth_match as sm
from tests.reference_outputs import Recorded, same


@pytest.fixture(scope="module")
def ref(oracle):
    return Recorded(oracle, __file__, oracle.ref_dbow2)


@pytest.mark.parametrize("k,L,scoring,weighting,levelsup", [(10, 3, 0, 0, 1), (10, 3, 0, 0, 4), (6, 4, 1, 1, 2), (4, 5, 5, 0, 3), (7, 3, 2, 2, 0),
                                                           (5, 3, 3, 3, 1), (9, 2, 4, 0, 1), (3, 6, 0, 0, 4), (20, 2, 5, 2, 1)])
def test_transform_matches_the_reference_code(ref, k, L, scoring, weighting, levelsup):
    voc = sm.make_vocabulary(k=k, L=L, seed=100 + k + L, scoring=scoring, weighting=weighting)
    feat = sm.make_voc_features(voc, n=600, seed=200 + k)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "voc.txt")
        ref.write_vocabulary_text(voc, path)
        R = ref.obj("RefVocabulary", lambda: ref.RefVocabulary(path))
    O = ref.Vocabulary(voc)
    assert R.words() == int(np.asarray(voc["is_leaf"]).sum())
    a, b = O.transform(feat, levelsup), R.transform(feat, levelsup)
    for key in ("word", "weight", "bow_id", "bow_val", "fv_node_id", "fv_node_ptr", "fv_feat"):
        assert same(a[key], b[key]), key
    if L - levelsup > 0:           # otherwise the reference leaves *nid untouched for non-root levels; both report the root
        assert same(a["node"], b["node"])
    assert len(a["bow_id"]) > 20
    O.close(); R.close()


def test_forb_distance_matches_the_reference_code(ref):
    rng = np.random.default_rng(0)
    A = rng.integers(0, 256, size=(200, 32), dtype=np.uint8); B = rng.integers(0, 256, size=(200, 32), dtype=np.uint8)
    B[:20] = A[:20]; B[20] = np.bitwise_not(A[20])
    for a, b in zip(A, B):
        assert ref.ref_forb_distance(a, b) == ref.descriptor_distance(a, b) == int(np.unpackbits(a ^ b).sum())
    assert ref.ref_forb_distance(A[20], B[20]) == 256 and ref.ref_forb_distance(A[0], B[0]) == 0
