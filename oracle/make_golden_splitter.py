"""Generate tests/golden/image_splitter.json by running the reference's own ImageSpliterTh (utils/util_image.py).

    RESSHIFT_REFERENCE=<path to the ResShift tree> python -m oracle.make_golden_splitter

Records, for every case the tiling tests check, the row / column starts the splitter computes and the tiles it yields
per batch (their (h, w) starts in latent units and the shape of the stacked patch).  Nothing here copies reference
source; it only imports and executes it.
"""
from __future__ import annotations

import json
import os
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
GOLD = ROOT / "tests" / "golden"

# (length, patch, stride) of tile_starts: every length in 1..69 and some larger ones, against these patch / stride pairs
STARTS_LENGTHS = list(range(1, 70)) + [100, 127, 128, 129, 200, 255, 256, 257, 300, 448, 500, 592, 1000]
STARTS_PATCHES = [(16, 16), (16, 12), (32, 28), (64, 64), (128, 112), (256, 224)]
# (h, w, patch, stride, sf, extra_bs) of plan_tiles, on a [2, 3, h, w] image
PLAN_CASES = [(75, 50, 32, 28, 4, 1), (148, 112, 128, 112, 4, 3), (64, 200, 64, 48, 4, 8),
              (40, 40, 64, 48, 4, 2), (592 // 4, 448 // 4, 128, 112, 4, 4), (512, 700, 256, 224, 1, 5)]


def main():
    ref = os.environ.get("RESSHIFT_REFERENCE")
    if not ref:
        raise SystemExit("set RESSHIFT_REFERENCE to the reference ResShift tree")
    sys.path[:0] = [str(ROOT / "oracle" / "_shims"), ref]
    from utils.util_image import ImageSpliterTh                  # noqa: E402  (reference)

    starts = []
    for n in STARTS_LENGTHS:
        for ps, st in STARTS_PATCHES:
            sp = ImageSpliterTh(torch.zeros(1, 1, n, max(n // 2, 1)), ps, st, sf=1)
            starts.append({"n": n, "patch": ps, "stride": st, "height_starts": sp.height_starts_list,
                           "width_starts": sp.width_starts_list})
    plans = []
    for (h, w, ps, st, sf, bs) in PLAN_CASES:
        sp = ImageSpliterTh(torch.zeros(2, 3, h, w), ps, st, sf=sf, extra_bs=bs)
        groups, shapes = [], []
        for pch, idx in sp:
            groups.append([[i[0] // sf, i[2] // sf] for i in idx])
            shapes.append([pch.shape[0], pch.shape[2], pch.shape[3]])
        plans.append({"h": h, "w": w, "patch": ps, "stride": st, "sf": sf, "bs": bs, "groups": groups,
                      "patch_shapes": shapes, "height_starts": sp.height_starts_list, "width_starts": sp.width_starts_list})
    GOLD.mkdir(parents=True, exist_ok=True)
    (GOLD / "image_splitter.json").write_text(json.dumps({"tile_starts": starts, "plan_tiles": plans}, separators=(",", ":")) + "\n")


if __name__ == "__main__":
    main()
