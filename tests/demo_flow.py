"""TEST INFRASTRUCTURE — the single-image flow of the reference's ``demo.py`` restated so that it runs without a
reference checkout: same steps, same module names — it imports the hot-path classes from the names the reference uses
(``src.smirk_encoder`` ...), which ``python -m smirk_b200.dropin`` aliases to smirk_b200 — and writes the same grid
image.  Each block cites the demo.py lines it follows.  tests/test_dropin_demo.py runs it on the GPU and, with the CPU
oracle in place of the native calls, without one.

    python -m smirk_b200.dropin tests/demo_flow.py --input_path x.png --checkpoint ck.pt --out_path out [--use_smirk_generator]
"""
import argparse
import os
import sys

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import dropin_support                                             # noqa: E402  (synthetic landmarks: the mediapipe stand-in)
from src.smirk_encoder import SmirkEncoder                        # noqa: E402  demo.py:5
from src.FLAME.FLAME import FLAME                                 # noqa: E402  demo.py:6
from src.renderer.renderer import Renderer                        # noqa: E402  demo.py:7

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--input_path", required=True)
    ap.add_argument("--device", default="cuda")
    ap.add_argument("--checkpoint", required=True)
    ap.add_argument("--out_path", default="output")
    ap.add_argument("--use_smirk_generator", action="store_true")
    ap.add_argument("--dump", default=None, help="also save the tensors of the run here (.pt), for stage-wise checks")
    ap.add_argument("--coords", default=None, help="masking samples (.npz: sampled_faces_indices, barycentric_coords) to use "
                                                   "instead of drawing them, e.g. those of another run's --dump")
    args = ap.parse_args()

    # demo.py:54-59 — encoder + checkpoint ingest (keys carry a `smirk_encoder.` prefix)
    smirk_encoder = SmirkEncoder().to(args.device)
    checkpoint = torch.load(args.checkpoint)
    smirk_encoder.load_state_dict({k.replace("smirk_encoder.", ""): v for k, v in checkpoint.items() if "smirk_encoder" in k})
    smirk_encoder.eval()
    if hasattr(smirk_encoder, "precision"):
        smirk_encoder.precision = int(os.environ.get("SMK_DEMO_PRECISION", "3"))
    if args.use_smirk_generator:                                    # demo.py:61-67
        from src.smirk_generator import SmirkGenerator
        smirk_generator = SmirkGenerator(in_channels=6, out_channels=3, init_features=32, res_blocks=5).to(args.device)
        smirk_generator.load_state_dict({k.replace("smirk_generator.", ""): v for k, v in checkpoint.items() if "smirk_generator" in k})
        smirk_generator.eval()
        if hasattr(smirk_generator, "precision"):
            smirk_generator.precision = 1
    flame = FLAME().to(args.device)                                 # demo.py:71-72
    renderer = Renderer().to(args.device)

    image = cv2.imread(args.input_path)                             # demo.py:78-81 (landmarks: synthetic stand-in)
    kpt = dropin_support.synthetic_landmarks(image.shape[1], image.shape[0])
    cropped_image = cv2.cvtColor(image, cv2.COLOR_BGR2RGB)          # demo.py:102-105 (no --crop)
    cropped_image = cv2.resize(cropped_image, (224, 224))
    cropped_image = torch.tensor(cropped_image).permute(2, 0, 1).unsqueeze(0).float() / 255.0
    cropped_image = cropped_image.to(args.device)

    outputs = smirk_encoder(cropped_image)                          # demo.py:107-114
    flame_output = flame.forward(outputs)
    renderer_output = renderer.forward(flame_output["vertices"], outputs["cam"], landmarks_fan=flame_output["landmarks_fan"],
                                       landmarks_mp=flame_output["landmarks_mp"])
    rendered_img = renderer_output["rendered_img"]
    grid = torch.cat([cropped_image, rendered_img], dim=3)          # demo.py:129
    dump = {"cropped_image": cropped_image, "outputs": outputs, "vertices": flame_output["vertices"], "rendered_img": rendered_img,
            "transformed_vertices": renderer_output["transformed_vertices"]}

    if args.use_smirk_generator:                                    # demo.py:133-169, masking on the GPU (smirk_b200.masking)
        from smirk_b200 import masking
        lm = kpt[:, :2].copy()                                      # the script masks in ORIGINAL image coordinates (demo.py:100,142)
        hull = cv2.convexHull(np.ascontiguousarray(lm.astype(np.int32)))
        hull_mask = np.ones((224, 224), np.uint8)
        cv2.fillConvexPoly(hull_mask, hull, 0)                      # datasets/base_dataset.py:9-15
        g = torch.Generator().manual_seed(77)
        face_probabilities = (torch.rand(flame.faces_tensor.shape[0], generator=g) > 0.5).float()
        rendered_mask = 1 - (rendered_img == 0).all(dim=1, keepdim=True).float()
        tv = renderer_output["transformed_vertices"]
        w = masking.face_weights(tv, flame.faces_tensor, face_probabilities)
        num = int(0.05 * 224 * 224)
        idx = torch.multinomial(w.cpu(), num, replacement=True, generator=g)
        u, v = torch.rand(num, generator=g), torch.rand(num, generator=g)
        o = u + v > 1
        u[o], v[o] = 1 - u[o], 1 - v[o]
        bary = torch.stack((1 - (u + v), u, v), 1)[None]
        if args.coords:                                             # the draws depend on the last bits of the weights
            c = np.load(args.coords)
            idx, bary = torch.from_numpy(c["sampled_faces_indices"]).long(), torch.from_numpy(c["barycentric_coords"]).float()
        npoints, _ = masking.mesh_based_mask_uniform_faces(tv, flame.faces_tensor, face_probabilities, mask_ratio=0.05,
                                                           coords={"sampled_faces_indices": idx, "barycentric_coords": bary})
        rbound = torch.tensor([num // 2])
        hull_t = torch.from_numpy(hull_mask).float()[None, None].to(args.device)
        masked_img = masking.masking_from_points(cropped_image, hull_t, npoints, rbound, wr=10, rendered_mask=rendered_mask,
                                                 flame_faces=flame.faces_tensor)
        smirk_generator_input = torch.cat([rendered_img, masked_img], dim=1)
        reconstructed_img = smirk_generator(smirk_generator_input)
        grid = torch.cat([grid, reconstructed_img], dim=3)
        dump.update(generator_input=smirk_generator_input, reconstructed_img=reconstructed_img, npoints=npoints,
                    sampled_faces_indices=idx, barycentric_coords=bary)

    grid_numpy = (grid.squeeze(0).permute(1, 2, 0).detach().cpu().numpy() * 255.0).astype(np.uint8)   # demo.py:170-182
    grid_numpy = cv2.cvtColor(grid_numpy, cv2.COLOR_BGR2RGB)
    os.makedirs(args.out_path, exist_ok=True)
    cv2.imwrite("%s/%s" % (args.out_path, args.input_path.split("/")[-1]), grid_numpy)
    if args.dump:
        torch.save({k: (v.cpu() if torch.is_tensor(v) else {kk: vv.cpu() for kk, vv in v.items()}) for k, v in dump.items()}, args.dump)
