"""ORACLE — TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the REFERENCE's own
Python classes (via oracle/ref_harness.py) in the build container.  Re-run: ``python -m oracle.make_golden``.

Every array stored here is an output of reference code (src/FLAME/FLAME.py, src/FLAME/lbs.py,
src/renderer/renderer.py + util.py, src/smirk_generator.py, src/smirk_encoder.py heads) on the
seeded inputs of smirk_b200/synth_inputs.py and the asset tree of smirk_b200/synth_assets.py.
Third-party pieces stubbed by the harness (pytorch3d rasteriser, timm backbones) are the Tier-B
restatements — the fixtures pin them only against regressions, not against upstream (unpinned).
"""
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
from smirk_b200 import synth_assets, synth_inputs  # noqa: E402
from oracle import ref_harness  # noqa: E402

GOLD = os.path.join(HERE, "..", "tests", "golden")
N = lambda t: t.detach().cpu().numpy()


def savez_lzma(path, **arrays):
    """Like np.savez_compressed, with LZMA members (np.load reads them): keeps render.npz under 1 MB."""
    import io
    import zipfile
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, a in arrays.items():
            buf = io.BytesIO()
            np.save(buf, a)
            z.writestr(k + ".npy", buf.getvalue())


def main():
    root = synth_assets.materialize(os.path.join(tempfile.gettempdir(), "smk_assets_golden"))
    with ref_harness.reference(root) as R, torch.no_grad():
        flame, rend = R.FLAME(), R.Renderer()
        # ---- FLAME ------------------------------------------------------------------------------
        out = {}
        p = synth_inputs.flame_params(4, 101)
        fo = flame.forward(p)
        out.update({"full/" + k: N(v) for k, v in fo.items()})
        p2 = synth_inputs.flame_params(2, 102)
        short = {"shape_params": p2["shape_params"][:, :100], "expression_params": p2["expression_params"][:, :20],
                 "pose_params": p2["pose_params"], "jaw_params": p2["jaw_params"]}
        out.update({"short/" + k: N(v) for k, v in flame.forward(short).items()})
        out.update({"zero/" + k: N(v) for k, v in
                    flame.forward(dict(p2), zero_expression=True, zero_shape=True, zero_pose=True).items()})
        # yaw sweep for the dynamic-contour LUT (FLAME.py:145-153), incl. |yaw| > 39 deg
        ps = synth_inputs.flame_params(8, 103)
        ps["pose_params"] = torch.tensor([[0.1, y, 0.05] for y in (-1.2, -0.69, -0.3, -0.01, 0.0, 0.2, 0.68, 1.3)])
        fs = flame.forward(ps)
        out["sweep/landmarks_fan"] = N(fs["landmarks_fan"])
        # C1: lbs() B=1 (BASELINE.json configs[0])
        p1 = synth_inputs.flame_params(1, 1001)
        betas = torch.cat([p1["shape_params"], p1["expression_params"]], 1)
        pose = torch.cat([p1["pose_params"], torch.zeros(1, 3), p1["jaw_params"], torch.zeros(1, 6)], 1)
        v, J = R.lbs.lbs(betas, pose, flame.v_template[None], flame.shapedirs, flame.posedirs, flame.J_regressor,
                         flame.parents, flame.lbs_weights)
        out["c1/verts"], out["c1/joints"] = N(v), N(J)
        np.savez_compressed(os.path.join(GOLD, "flame.npz"), **out)
        # ---- Renderer ---------------------------------------------------------------------------
        pr = synth_inputs.flame_params(2, 201)
        fr = flame.forward(pr)
        ro = rend.forward(fr["vertices"], pr["cam"], landmarks_fan=fr["landmarks_fan"], landmarks_mp=fr["landmarks_mp"])
        # raw rasteriser outputs through the same stubbed call the reference makes (renderer.py:184-193)
        from oracle import render_ref
        rr = render_ref.render_forward_ref(render_ref.RenderConstants(root), fr["vertices"], pr["cam"])
        assert torch.equal(ro["transformed_vertices"], rr["transformed_vertices"])
        savez_lzma(os.path.join(GOLD, "render.npz"),
                   vertices=N(fr["vertices"]), cam=N(pr["cam"]),
                   rendered_img=N(ro["rendered_img"]), transformed_vertices=N(ro["transformed_vertices"]),
                   landmarks_fan=N(ro["landmarks_fan"]), landmarks_mp=N(ro["landmarks_mp"]),
                   pix_to_face=N(rr["pix_to_face"]).astype(np.int32), bary=N(rr["bary"]),
                   faces=N(rend.faces[0]).astype(np.int16))
        # ---- Generator --------------------------------------------------------------------------
        gen = R.SmirkGenerator(in_channels=6, out_channels=3, init_features=32, res_blocks=5).eval()
        gen.load_state_dict(synth_inputs.random_state_dict(gen.state_dict(), seed=7))
        x = torch.cat([ro["rendered_img"][:1], synth_inputs.masked_images(1, 301)], 1)
        y = gen(x)
        np.savez_compressed(os.path.join(GOLD, "generator.npz"), y_sub=N(y[:, :, ::4, ::4]),
                            y_mean=N(y.mean((2, 3))), y_rows=N(y[:, :, 100:102, :]),
                            n_keys=np.int64(len(gen.state_dict())))
        # ---- Encoder (reference heads over the restated timm backbones) ---------------------------
        enc = R.SmirkEncoder().eval()
        enc.load_state_dict(synth_inputs.random_state_dict(enc.state_dict(), seed=7))
        eo = enc(synth_inputs.images(2, 401))
        np.savez_compressed(os.path.join(GOLD, "encoder.npz"), **{k: N(v) for k, v in eo.items()},
                            n_keys=np.int64(len(enc.state_dict())))
        for k, v in eo.items():
            print(k, v.shape, float(v.abs().mean()), float(v.abs().max()))
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == "__main__":
    main()
