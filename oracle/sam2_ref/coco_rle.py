"""ORACLE (test infrastructure only). Restatement of upstream sam2/utils/amg.py coco_encode_rle, which converts an
uncompressed RLE with pycocotools (mask_utils.frPyObjects), i.e. maskApi.c rleToString, and of its inverse rleFrString
for round trips. pycocotools itself is not a dependency.
"""
from __future__ import annotations

from typing import Any, Dict, List


def counts_to_string(counts: List[int]) -> str:
    """maskApi.c rleToString: each count minus the count two places back (from the fourth on) in signed 5-bit groups,
    least significant first, 0x20 = more groups follow, offset by 48."""
    out = []
    for i, c in enumerate(counts):
        x = int(c) - (int(counts[i - 2]) if i > 2 else 0)
        more = True
        while more:
            ch = x & 0x1F
            x >>= 5  # Python's >> on ints is arithmetic, as on C's signed long
            more = (x != -1) if (ch & 0x10) else (x != 0)
            if more:
                ch |= 0x20
            out.append(chr(ch + 48))
    return "".join(out)


def string_to_counts(s: str) -> List[int]:
    """maskApi.c rleFrString."""
    counts: List[int] = []
    p = 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            c = ord(s[p]) - 48
            x |= (c & 0x1F) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)
        if len(counts) > 2:
            x += counts[-2]
        counts.append(x)
    return counts


def coco_encode_rle(uncompressed_rle: Dict[str, Any]) -> Dict[str, Any]:
    """upstream coco_encode_rle: {"size": [h, w], "counts": str}"""
    h, w = uncompressed_rle["size"]
    return {"size": [h, w], "counts": counts_to_string(uncompressed_rle["counts"])}


def coco_decode_rle(rle: Dict[str, Any]) -> Dict[str, Any]:
    """the uncompressed RLE a compressed one encodes"""
    h, w = rle["size"]
    return {"size": [h, w], "counts": string_to_counts(rle["counts"])}
