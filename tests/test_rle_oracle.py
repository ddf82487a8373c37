"""CPU: the oracle's run-length encodings. mask_to_rle (upstream mask_to_rle_pytorch) against a direct column-major
restatement, and the COCO string codec (pycocotools' rleToString / rleFrString) against hand-worked vectors and in
round trips, including negative deltas and values that need five or more characters."""
import numpy as np
import pytest

from oracle.sam2_ref import amg as up
from oracle.sam2_ref.coco_rle import coco_decode_rle, coco_encode_rle, counts_to_string, string_to_counts


def runs_column_major(mask):
    """counts by walking the pixels in column-major order: the zeros first, then alternating runs"""
    flat = [bool(v) for v in np.asarray(mask).T.reshape(-1)]
    counts, cur, run = [], False, 0
    for v in flat:
        if v != cur:
            counts.append(run)
            cur, run = v, 0
        run += 1
    counts.append(run)
    return counts


def sample_masks(rng):
    out = []
    for H, W in [(1, 1), (1, 7), (7, 1), (5, 9), (33, 40), (64, 65)]:
        out += [np.zeros((H, W), bool), np.ones((H, W), bool), rng.uniform(size=(H, W)) < 0.5,
                rng.uniform(size=(H, W)) < 0.05]
        first = np.zeros((H, W), bool)
        first[0, 0] = True
        last = np.zeros((H, W), bool)
        last[-1, -1] = True
        alt = (np.arange(H * W) % 2 == 0).reshape(W, H).T  # column-major alternation from a set pixel
        out += [first, last, alt]
    return out


def test_encoder_hand_worked_vectors():
    assert counts_to_string([0, 40]) == "0X1"
    assert counts_to_string([5, 2, 3, 1]) == "523O"
    assert string_to_counts("0X1") == [0, 40]
    assert string_to_counts("523O") == [5, 2, 3, 1]
    assert coco_encode_rle({"size": [4, 10], "counts": [0, 40]}) == {"size": [4, 10], "counts": "0X1"}


def test_mask_to_rle_is_column_major_runs():
    rng = np.random.default_rng(0)
    for mask in sample_masks(rng):
        rle = up.mask_to_rle(mask)
        assert rle["size"] == list(mask.shape)
        assert rle["counts"] == runs_column_major(mask)
        assert sum(rle["counts"]) == mask.size
        assert up.area_from_rle(rle) == int(mask.sum())
        np.testing.assert_array_equal(up.rle_to_mask(rle), mask)
    H, W = 5, 9
    alt = (np.arange(H * W) % 2 == 0).reshape(W, H).T
    assert len(up.mask_to_rle(alt)["counts"]) == H * W + 1  # the most counts a mask can have


@pytest.mark.parametrize("seed", range(4))
def test_coco_round_trip_random_masks(seed):
    rng = np.random.default_rng(seed)
    for mask in sample_masks(rng):
        rle = up.mask_to_rle(mask)
        enc = coco_encode_rle(rle)
        assert isinstance(enc["counts"], str) and all(48 <= ord(c) < 48 + 64 for c in enc["counts"])
        assert coco_decode_rle(enc) == rle


def test_coco_round_trip_large_and_negative_deltas():
    rng = np.random.default_rng(7)
    # counts whose deltas to two places back are negative, zero, and need 1..7 five-bit groups
    vals = [0, 1, 15, 16, 31, 32, 511, 512, 1 << 15, (1 << 20) + 3, (1 << 25) - 1, (1 << 30) + 17, (1 << 31) - 2]
    for _ in range(200):
        counts = [int(v) for v in rng.choice(vals, size=rng.integers(1, 12))]
        s = counts_to_string(counts)
        assert string_to_counts(s) == counts
    # a delta of -(2^30) (cnts[3] - cnts[1]) takes 7 characters; 2^31 - 2 as the first count takes 7 as well
    s = counts_to_string([0, (1 << 30) + 1, 0, 1])
    assert string_to_counts(s) == [0, (1 << 30) + 1, 0, 1]
    assert len(counts_to_string([(1 << 31) - 2])) == 7
    assert len(counts_to_string([0, 1 << 30, 0, 0])) - len(counts_to_string([0, 1 << 30, 0])) == 7
    assert counts_to_string([3, 4, 3]) == "343"  # i == 2 is not differenced
    assert counts_to_string([3, 4, 3, 4]) == "3430"  # i == 3 is: 4 - 4
