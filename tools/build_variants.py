#!/usr/bin/env python
"""Cross-compile tuning builds of libskychunk.so into tools/bin/ (they travel to the GPU box; SKYCHUNK_LIB selects one)."""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from skyplane_b200 import build  # noqa: E402

VARIANTS = {
    "pa10_r3": {"SKY_PARSERS": 10, "SKY_RING_EXTRA": 3},
    "pa12_r2": {"SKY_PARSERS": 12, "SKY_RING_EXTRA": 2},  # the default build
    "pa13_r1": {"SKY_PARSERS": 13, "SKY_RING_EXTRA": 1},
}

if __name__ == "__main__":
    names = sys.argv[1:] or list(VARIANTS)
    out = ROOT / "tools" / "bin"
    out.mkdir(exist_ok=True)
    for n in names:
        print(build.build_variant(out / f"libskychunk_{n}.so", VARIANTS[n]))
