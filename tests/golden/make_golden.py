"""Generate the committed golden fixtures from a checkout of the reference project (needs no GPU).

* smoke_*.npy : the reference's in-repo snapshot PNGs (vello_tests/snapshots/smoke/*.png; the
  other snapshot directories are git-LFS pointers) decoded to RGBA8 arrays. They pin the oracle
  (tests/test_oracle_golden.py); recipes: vello_tests/tests/smoke_snapshots.rs:17-52,
  vello_tests/tests/regression.rs:33-210, vello_tests/tests/known_issues.rs:21-52.
* tiger_paths.json.gz : the Ghostscript tiger (examples/assets/Ghostscript_Tiger.svg, the asset
  BASELINE.json configs C1/C2 name) reduced to the draw list `pico_svg` produces
  (examples/scenes/src/pico_svg.rs:134-195): per <path> the fill / stroke colours, stroke width
  and the path data string. The SVG itself is not copied.

Usage: python tests/golden/make_golden.py <reference checkout>
"""
import gzip
import json
import os
import re
import sys
import xml.etree.ElementTree as ET

import numpy as np
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))


def main(ref):
    smoke = os.path.join(ref, "vello_tests/snapshots/smoke")
    for name in ["filled_square", "filled_circle", "layer_size", "gradient_color_alpha_premultiplied",
                 "gradient_color_alpha_unpremultiplied", "data_image_roundtrip"]:
        a = np.array(Image.open(os.path.join(smoke, name + ".png")).convert("RGBA"))
        np.save(os.path.join(HERE, f"smoke_{name}.npy"), a)
        print(name, a.shape)
    tree = ET.parse(os.path.join(ref, "examples/assets/Ghostscript_Tiger.svg"))
    root = tree.getroot()
    ns = re.match(r"\{.*\}", root.tag).group(0)
    items = []

    def rec(node, fill):
        tag = node.tag.replace(ns, "")
        f = node.get("fill")
        if f is not None:
            fill = None if f == "none" else f
        if tag in ("g", "svg"):
            assert node.get("transform") is None
            for ch in node:
                rec(ch, fill)
        elif tag == "path":
            it = {"d": node.get("d"), "fill": fill}
            for k in ("fill-opacity", "opacity", "stroke", "stroke-width", "stroke-opacity"):
                if node.get(k) is not None:
                    it[k] = node.get(k)
            items.append(it)

    # the document element only contributes the default black fill (pico_svg.rs:106-108)
    for ch in root:
        rec(ch, "#000")
    out = {"viewBox": root.get("viewBox"), "items": items}
    with gzip.open(os.path.join(HERE, "tiger_paths.json.gz"), "wt", compresslevel=9) as f:
        json.dump(out, f, separators=(",", ":"))
    print("tiger items", len(items))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
