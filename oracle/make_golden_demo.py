"""ORACLE — TEST INFRASTRUCTURE ONLY.  Generates tests/golden/demo.npz with the REFERENCE's own classes on the CPU —
third-party pieces (timm, pytorch3d, skimage, mediapipe) replaced by the stand-ins of oracle/ref_harness.py and
tests/dropin_support.py — on the synthetic input image and synthetic checkpoint of tests/dropin_support.py.  Needs a
reference checkout (``SMIRK_REFERENCE``): ``python -m oracle.make_golden_demo``.

Stored:
  grid            the grid the reference's own, unmodified ``demo.py`` writes (demo.py:170-182) without
                  ``--use_smirk_generator`` (cropped image | rendered mesh);
  grid_generator  the grid tests/demo_flow.py writes with ``--use_smirk_generator`` (cropped image | rendered mesh |
                  SmirkGenerator output) when its ``src.*`` imports resolve to the reference's classes; its masking step
                  is the CPU oracle (tests/dropin_support.py), as in the test that compares against it;
  generator_sampled_faces_indices, generator_barycentric_coords
                  the masking samples that run drew.  The draws depend on the last bits of the face weights, which vary
                  with the CPU, so the test replays these instead of drawing its own.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import cv2
    import dropin_support as ds
    from smirk_b200 import synth_assets
    from oracle import ref_harness
    work = tempfile.mkdtemp(prefix="smk_demo_golden_")
    root = synth_assets.materialize(os.path.join(work, "assets_root"))
    img = ds.synthetic_image(os.path.join(work, "face.png"))
    grids, dump = {}, os.path.join(work, "dump.pt")
    for key, script, generator in (("grid", os.path.join(ref_harness.REF, "demo.py"), False),
                                   ("grid_generator", os.path.join(ROOT, "tests", "demo_flow.py"), True)):
        ck = ds.write_checkpoint(os.path.join(work, key + ".pt"), with_generator=generator)
        out = os.path.join(work, "out_" + key)
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tests", "dropin_support.py"), "--mode", "reference", "--script", script,
                               "--reference-root", ref_harness.REF, "--cwd", root, "--", "--input_path", img, "--device", "cpu",
                               "--checkpoint", ck, "--out_path", out] + (["--use_smirk_generator", "--dump", dump] if generator else []))
        grids[key] = cv2.imread(os.path.join(out, "face.png"))
    import torch
    t = torch.load(dump)
    grids["generator_sampled_faces_indices"] = t["sampled_faces_indices"].numpy().astype(np.int32)
    grids["generator_barycentric_coords"] = t["barycentric_coords"].numpy().astype(np.float32)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "demo.npz"), **grids)
    print("demo.npz:", {k: g.shape for k, g in grids.items()},
          "rendered coverage %.3f" % float((grids["grid"][:, 224:] > 0).any(-1).mean()))


if __name__ == "__main__":
    main()
