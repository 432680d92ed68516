"""How much of fast_kernel's exact-score work the cheap reject leaves, on the bench input (CPU only).

For the 8 images of synth.stereo_pair(2024, 0, 0..3) at KITTI shape, the pyramid comes from the oracle port
(oracle.PortExtractor).  Per level, over the FAST detection domain [19, w-19) x [19, h-19), it counts at threshold t:
  reject4   the kernel's reject: for each of the 4 even antipodal ring pairs (0,8) (2,10) (4,12) (6,14) one of the two
            differs from the centre by more than t, either polarity (fast_kernel phase 1a; the kernel's carry-based flag
            can add rare false keeps, not counted here)
  polar8    a polarity-aware reject on all 8 antipodal pairs: every pair has a pixel > I_p + t, or every pair a pixel
            < I_p - t
  corner    true FAST-9 corners at t (9 contiguous ring pixels all > I_p + t or all < I_p - t)
as the share of domain pixels kept and of aligned 4-pixel words (x // 4) holding at least one kept domain pixel.  "all" is
weighted by pixel count (sums over levels).  A word-granular scoring pass scores 4 pixels per kept word; a pixel-granular
one scores only the kept pixels.
usage: python tools/fast_survivors.py [--th 20] [--pairs 4]  -> one JSON line."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle_lib as O                                            # noqa: E402
from orb_slam2_b200 import synth                                              # noqa: E402

EDGE = 19
RX = [0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1]
RY = [3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3]


def level_counts(img, t):
    h, w = img.shape
    I = img.astype(np.int16)
    c = I[EDGE:h - EDGE, EDGE:w - EDGE]
    d = [I[EDGE + dy:h - EDGE + dy, EDGE + dx:w - EDGE + dx] - c for dx, dy in zip(RX, RY)]
    hi = [x > t for x in d]
    lo = [x < -t for x in d]
    big = [a | b for a, b in zip(hi, lo)]
    reject4 = np.logical_and.reduce([big[j] | big[j + 8] for j in (0, 2, 4, 6)])
    polar8 = np.logical_and.reduce([hi[j] | hi[j + 8] for j in range(8)]) | np.logical_and.reduce([lo[j] | lo[j + 8] for j in range(8)])
    corner = np.zeros_like(reject4)
    for k in range(16):
        corner |= np.logical_and.reduce([hi[(k + j) % 16] for j in range(9)])
        corner |= np.logical_and.reduce([lo[(k + j) % 16] for j in range(9)])
    word = (np.arange(EDGE, w - EDGE) // 4)[None, :]               # aligned word of each domain column
    nwords = int(np.unique(word).size) * c.shape[0]
    out = {"pixels": int(c.size), "words": nwords}
    for name, m in (("reject4", reject4), ("polar8", polar8), ("corner", corner)):
        kept_words = 0
        for row in m:
            kept_words += int(np.unique(word[0][row]).size)
        out[name] = {"pixels_kept": int(m.sum()), "words_kept": kept_words}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--th", type=int, default=20, help="FAST threshold (iniThFAST of the bench: 20)")
    ap.add_argument("--pairs", type=int, default=4, help="stereo pairs of the bench input (2 images each)")
    a = ap.parse_args()
    P = O.PortExtractor(2000)
    tot = {}
    for p in range(a.pairs):
        for img in synth.stereo_pair(2024, 0, p, *synth.KITTI)[:2]:
            P(img)
            for l in range(8):
                r = level_counts(P.level(l), a.th)
                acc = tot.setdefault(l, {"pixels": 0, "words": 0})
                acc["pixels"] += r["pixels"]; acc["words"] += r["words"]
                for k in ("reject4", "polar8", "corner"):
                    s = acc.setdefault(k, {"pixels_kept": 0, "words_kept": 0})
                    s["pixels_kept"] += r[k]["pixels_kept"]; s["words_kept"] += r[k]["words_kept"]
    allc = {"pixels": sum(v["pixels"] for v in tot.values()), "words": sum(v["words"] for v in tot.values())}
    for k in ("reject4", "polar8", "corner"):
        allc[k] = {f: sum(v[k][f] for v in tot.values()) for f in ("pixels_kept", "words_kept")}

    def shares(v):
        return {k: {"words_kept": v[k]["words_kept"] / v["words"], "pixels_kept": v[k]["pixels_kept"] / v["pixels"]}
                for k in ("reject4", "polar8", "corner")}
    print(json.dumps({"what": "fast_kernel reject survivors on the bench input", "threshold": a.th, "images": 2 * a.pairs,
                      "all": shares(allc), "levels": {l: shares(v) for l, v in tot.items()}}))


if __name__ == "__main__":
    main()
