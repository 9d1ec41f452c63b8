"""TEST INFRASTRUCTURE — everything needed to run one of the reference's entry scripts (demo.py) end to end without
its third-party stack: stub ``skimage.transform`` / ``mediapipe`` / ``albumentations`` modules, a synthetic
``SMIRK_em1.pt``-style checkpoint (``smirk_encoder.`` / ``smirk_generator.`` key prefixes, demo.py:55-58,65-66), a
synthetic input image, and a subprocess runner with three modes:

  reference      the REFERENCE's own classes (src/smirk_encoder.py, FLAME.py, renderer.py, smirk_generator.py) with the
                 oracle's stand-ins for timm / pytorch3d (oracle/ref_harness.py) on the CPU           -> the golden run
  dropin         ``python -m smirk_b200.dropin <script>``: the four hot-path modules replaced by smirk_b200 (needs a GPU)
  dropin-oracle  like dropin, but the native forwards of the smirk_b200 classes are patched HERE, in test code, to
                 evaluate the CPU oracle: exercises the drop-in surface (aliasing, constructors, checkpoint ingest,
                 dict keys, attribute access from the script) on a machine without a GPU.  Never shipped.

In the reference and dropin-oracle modes the smirk_b200.masking calls of tests/demo_flow.py evaluate the CPU oracle too.

    python tests/dropin_support.py --mode reference --script <reference checkout>/demo.py --cwd <asset root> -- <script args>
    python tests/dropin_support.py --mode dropin-oracle --script tests/demo_flow.py --cwd <asset root> -- <script args>
"""
import argparse
import os
import runpy
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


# ------------------------------------------------------------------------------------------------ inputs
def synthetic_image(path, size=256, seed=3):
    """A smooth colour field with a face-like ellipse (uint8 BGR png)."""
    import cv2
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:size, 0:size].astype(np.float64) / size
    img = np.stack([0.5 + 0.4 * np.sin(6 * x + 1), 0.5 + 0.4 * np.cos(5 * y), 0.5 + 0.3 * np.sin(4 * (x + y))], -1)
    e = ((x - 0.5) / 0.28) ** 2 + ((y - 0.52) / 0.36) ** 2 < 1
    img[e] = 0.75 * img[e] + 0.25 * np.array([0.55, 0.62, 0.8])
    img = img + rng.normal(0, 0.02, img.shape)
    cv2.imwrite(path, (np.clip(img, 0, 1) * 255).astype(np.uint8))
    return path


def synthetic_landmarks(width, height, n=478):
    """Deterministic stand-in for mediapipe's 478 face landmarks: rings of points inside the face ellipse."""
    k = np.arange(n)
    r = 0.15 + 0.85 * ((k * 37) % 101) / 100.0
    t = 2 * np.pi * ((k * 61) % 89) / 89.0
    x = (0.5 + 0.26 * r * np.cos(t)) * width
    y = (0.52 + 0.34 * r * np.sin(t)) * height
    return np.stack([x, y, 0.01 * np.cos(t)], 1)


def write_checkpoint(path, with_generator=True, seed=7):
    """Synthetic checkpoint in the reference's file format (demo.py:55-58,65-66): one flat dict, keys prefixed with the
    sub-model name.  Key names come from the smirk_b200 mirrors, whose layout is the reference's (timm names)."""
    import torch
    import smirk_b200
    from smirk_b200 import synth_inputs
    enc = smirk_b200.SmirkEncoder()
    ck = {"smirk_encoder." + k: v for k, v in synth_inputs.random_state_dict(enc.state_dict(), seed=seed).items()}
    if with_generator:
        gen = smirk_b200.SmirkGenerator(6, 3, 32, 5)
        ck.update({"smirk_generator." + k: v for k, v in synth_inputs.random_state_dict(gen.state_dict(), seed=seed).items()})
    torch.save(ck, path)
    return path


# ------------------------------------------------------------------------------------------------ stubs
def install_third_party_stubs():
    """skimage.transform (estimate_transform, warp), mediapipe (+ tasks.python.vision), albumentations."""
    from smirk_b200 import crop
    from oracle import warp_ref

    def warp(image, inverse_map, output_shape=None, preserve_range=False, **kw):
        M = np.asarray(inverse_map.params if hasattr(inverse_map, "params") else inverse_map, np.float64)
        out = warp_ref.warp_ref(np.asarray(image), M, tuple(output_shape)).astype(np.float64)
        return out if preserve_range else out / 255.0

    sk = types.ModuleType("skimage")
    tr = types.ModuleType("skimage.transform")
    tr.estimate_transform, tr.warp, tr.SimilarityTransform = crop.estimate_transform, warp, crop.SimilarityTransform
    sk.transform = tr
    sys.modules.update({"skimage": sk, "skimage.transform": tr})
    sys.modules.setdefault("albumentations", types.ModuleType("albumentations"))
    # OpenCV >= 4.9 rejects the non-contiguous slice datasets/base_dataset.py:10-11 hands to convexHull (the reference's
    # pinned OpenCV copied it silently): an environment shim like ref_harness's NumPy-2 aliases, not a change of behaviour
    import cv2
    if not getattr(cv2.convexHull, "_smk_contig", False):
        orig = cv2.convexHull
        def convex_hull(points, *a, **k):
            return orig(np.ascontiguousarray(points), *a, **k)
        convex_hull._smk_contig = True
        cv2.convexHull = convex_hull

    class _Image:
        def __init__(self, image_format=None, data=None):
            self.data = data
            self.height, self.width = data.shape[:2]

    class _Detector:
        def detect(self, image):
            pts = synthetic_landmarks(image.width, image.height)
            lms = [types.SimpleNamespace(x=p[0] / image.width, y=p[1] / image.height, z=p[2]) for p in pts]
            return types.SimpleNamespace(face_landmarks=[lms])

    mp = types.ModuleType("mediapipe")
    mp.Image, mp.ImageFormat = _Image, types.SimpleNamespace(SRGB=1)
    tasks = types.ModuleType("mediapipe.tasks")
    py = types.ModuleType("mediapipe.tasks.python")
    vision = types.ModuleType("mediapipe.tasks.python.vision")
    py.BaseOptions = lambda **kw: types.SimpleNamespace(**kw)
    vision.FaceLandmarkerOptions = lambda **kw: types.SimpleNamespace(**kw)
    vision.FaceLandmarker = types.SimpleNamespace(create_from_options=lambda options: _Detector())
    py.vision, tasks.python, mp.tasks = vision, py, tasks
    sys.modules.update({"mediapipe": mp, "mediapipe.tasks": tasks, "mediapipe.tasks.python": py, "mediapipe.tasks.python.vision": vision})


def patch_native_with_oracle(asset_root):
    """dropin-oracle mode: replace the C-ABI calls of the four smirk_b200 modules by the CPU oracle (test code only)."""
    import torch
    import smirk_b200.smirk_encoder as E
    import smirk_b200.flame as F
    import smirk_b200.renderer as R
    import smirk_b200.smirk_generator as G
    from oracle import encoder_ref, flame_ref, render_ref, generator_ref
    fc, rc = flame_ref.FlameConstants(asset_root), render_ref.RenderConstants(asset_root)

    def enc_run(self, img):
        if self.training:
            raise RuntimeError("train mode")
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        o = encoder_ref.encoder_forward_ref(sd, img.float(), n_exp=self.n_exp)
        return [torch.cat([o["pose_params"], o["cam"]], 1), o["shape_params"],
                torch.cat([o["expression_params"], o["eyelid_params"], o["jaw_params"]], 1)]

    def flame_lbs(self, betas, full_pose, eyelid=None):
        ne = self.n_exp
        p = {"shape_params": betas[:, :-ne], "expression_params": betas[:, -ne:], "pose_params": full_pose[:, :3],
             "neck_pose_params": full_pose[:, 3:6], "jaw_params": full_pose[:, 6:9], "eye_pose_params": full_pose[:, 9:15]}
        if eyelid is not None:
            p["eyelid_params"] = eyelid
        return flame_ref.flame_forward_ref(fc, p)

    def render_full(self, vertices, cam_params, raw=True, **landmarks):
        return render_ref.render_forward_ref(rc, vertices.float(), cam_params.float(), **landmarks)

    def gen_forward(self, x):
        return generator_ref.generator_forward_ref({k: v.detach() for k, v in self.state_dict().items()}, x.float(), res_blocks=self._cfg[3])

    E.SmirkEncoder._run = enc_run
    F.FLAME.run_lbs = flame_lbs
    R.Renderer.render_full = render_full
    G.SmirkGenerator.forward = gen_forward
    import smirk_b200._lib as L
    L.require_cuda = lambda t, name: None


def patch_masking_with_oracle():
    """The three smirk_b200.masking calls tests/demo_flow.py makes, evaluated by the CPU oracle (test code only), so the
    flow's generator branch runs on a machine without a GPU — on the drop-in classes and on the reference's alike."""
    import smirk_b200.masking as M
    from oracle import masking_ref

    def face_weights(tv, faces, face_probabilities):
        return masking_ref.face_probabilities_ref(tv.float(), faces, face_probabilities.float())

    def mesh_based_mask_uniform_faces(tv, faces, face_probabilities, mask_ratio=0.1, coords=None, IMAGE_SIZE=224):
        idx, bary = coords["sampled_faces_indices"], coords["barycentric_coords"]
        return masking_ref.points_from_coords_ref(tv.float(), faces, idx, bary, IMAGE_SIZE), coords

    def masking_from_points(img, mask, npoints, rbound, wr=15, rendered_mask=None, flame_faces=None, **kw):
        extra = img * masking_ref.point_mask_ref(npoints, rbound, img.shape[-1])
        return masking_ref.masking_ref(img, mask, extra, wr, rendered_mask=rendered_mask)

    M.face_weights, M.mesh_based_mask_uniform_faces, M.masking_from_points = face_weights, mesh_based_mask_uniform_faces, masking_from_points


# ------------------------------------------------------------------------------------------------ runner
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", required=True, choices=["reference", "dropin", "dropin-oracle"])
    ap.add_argument("--script", required=True)
    ap.add_argument("--cwd", required=True, help="asset root (the scripts use relative asset paths)")
    ap.add_argument("--reference-root", default=None, help="checkout whose `src` package the script imports (default: the script's directory)")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("rest", nargs=argparse.REMAINDER)
    a = ap.parse_args()
    rest = a.rest[1:] if a.rest and a.rest[0] == "--" else a.rest
    import torch
    sys.dont_write_bytecode = True
    ref_root = os.path.abspath(a.reference_root or os.path.dirname(os.path.abspath(a.script)))
    install_third_party_stubs()
    os.chdir(a.cwd)
    if a.mode == "reference":
        from oracle import ref_harness
        ref_harness._install_stubs()
        sys.path.insert(0, ref_root)
    else:
        from smirk_b200 import dropin
        dropin.install(ref_root)
        if a.mode == "dropin-oracle":
            patch_native_with_oracle(a.cwd)
    if a.mode != "dropin":
        patch_masking_with_oracle()
    # The reference's demo.py draws its masking samples from torch's global RNG (masking.py:160-162,84-96; demo.py:151-152)
    # after building the models, whose constructors consume a class-dependent number of draws.  Re-seed at the first
    # masking call so the reference classes and the drop-in classes see the same sample stream.
    if os.path.isfile(os.path.join(ref_root, "src", "utils", "masking.py")):
        import src.utils.masking as M
        load_prob = M.load_probabilities_per_FLAME_triangle

        def seeded_load(*args, **kw):
            torch.manual_seed(a.seed)
            return load_prob(*args, **kw)
        M.load_probabilities_per_FLAME_triangle = seeded_load
    sys.argv = [a.script] + rest
    with torch.no_grad():
        runpy.run_path(a.script, run_name="__main__")


if __name__ == "__main__":
    main()
