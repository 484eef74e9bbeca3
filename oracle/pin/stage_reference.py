"""Stage the reference's Python packages where a GPU machine without the reference checkout can import them:
<reference>/{pyramid_dit,video_vae,diffusion_schedulers,trainer_misc} (+ the top-level utils.py they import) -> oracle/_ref/
(git-ignored, never committed).

TEST / BASELINE INFRASTRUCTURE, run by hand.  What reads the staged copy through oracle/pin/ref_shim.py: make_golden.py's GPU
fixture (`python oracle/pin/make_golden.py dropin`) and bench.py's optional `gpu_eager_baseline` leg.  No test and no product
module needs it.  Nothing is edited: files are copied byte for byte (checked below).

    python oracle/pin/stage_reference.py /path/to/Pyramid-Flow
"""
from __future__ import annotations

import filecmp
import shutil
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
DST = ROOT / "oracle" / "_ref"
PACKAGES = ("pyramid_dit", "video_vae", "diffusion_schedulers", "trainer_misc")
TOP_FILES = ("utils.py",)          # video_vae/modeling_causal_conv.py:11 imports the context-parallel helpers from it


def stage(src: Path, verbose: bool = True) -> None:
    if not (src / "pyramid_dit").is_dir():
        raise SystemExit(f"[stage_reference] {src} is not a Pyramid-Flow checkout (no pyramid_dit/)")
    DST.mkdir(parents=True, exist_ok=True)
    n = 0
    for pkg in PACKAGES:
        for f in (src / pkg).rglob("*.py"):
            out = DST / f.relative_to(src)
            out.parent.mkdir(parents=True, exist_ok=True)
            if not out.exists() or not filecmp.cmp(f, out, shallow=False):
                shutil.copyfile(f, out)
            n += 1
    for name in TOP_FILES:
        if not (DST / name).exists() or not filecmp.cmp(src / name, DST / name, shallow=False):
            shutil.copyfile(src / name, DST / name)
        n += 1
    (DST / "STAGED_FROM").write_text(f"{src} (unmodified copy of {', '.join(PACKAGES)}; {n} files)\n")
    if verbose:
        print(f"[stage_reference] {n} files -> {DST}")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    stage(Path(sys.argv[1]).resolve())
