"""TEST INFRASTRUCTURE ONLY.  Golden fixture for the mask pre/post-processing (SURVEY §8f rank 3): runs the UNMODIFIED
reference code - networks/volumetric_avatar/face_parcing.py FaceParsing.forward (:55-81) and notebooks/infer.py
InferenceWrapper.get_mask (:649-684) - in this container with the seeded stand-in networks of oracle/stub_nets.py plugged in
where the external BiSeNet / MODNet checkouts would be, and records inputs and outputs:

    python -m oracle.make_golden_masks        # writes tests/golden/masks.pt
"""
from __future__ import annotations

import pathlib
import sys
import types

import numpy as np
import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
GOLD = ROOT / "tests" / "golden"


def parsing_input(h, w, seed):
    """the seeded test image batch (2,3,h,w): white noise, sample 0 replaced by a smooth frame when the image is square"""
    from oracle import frames as FR

    x = torch.rand(2, 3, h, w, generator=torch.Generator().manual_seed(seed))
    if h == w:
        x[0] = FR.frame(h, 41, "smooth")[0]
    return x


def main():
    import oracle.ref_harness as H
    from oracle import frames as FR
    from oracle.stub_nets import StubBiSeNet, StubMODNet

    H.install_stubs()
    sys.modules["repos.face_par_off.model"].BiSeNet = StubBiSeNet
    from networks.volumetric_avatar.face_parcing import FaceParsing  # the reference class, unmodified
    import notebooks.infer as ref_infer

    out = {}
    # inputs are regenerated from their seeds by the tests (torch's CPU generator is machine-independent); only outputs are stored
    for name, (h, w), seed in (("p512", (512, 512), 11), ("p256", (256, 256), 12), ("p300x400", (300, 400), 13)):
        fp = FaceParsing(None, device="cpu", project_dir=str(ROOT))
        x = parsing_input(h, w, seed)
        with torch.no_grad():
            masks = fp.forward(x)
            # the intermediate tensors of the same call sequence (face_parcing.py:57-60), strided samples only
            xn = (x - fp.mean[None, :, None, None]) / fp.std[None, :, None, None]
            x512 = torch.nn.functional.interpolate(xn, size=(512, 512), mode="bilinear")
        # the masks whole (bit-packed uint8 tensors), the resized input strided: the fixture stays under 1 MB
        out[name] = {"seed": seed, "shape": (h, w), "masks_packed": [torch.from_numpy(np.packbits(m.numpy().astype(np.uint8))) for m in masks],
                     "masks_sum": [int(m.sum()) for m in masks], "x512_s16": x512[:, :, ::16, ::16].clone()}
    fake_self = types.SimpleNamespace(modnet=StubMODNet())
    for name, (h, w), seed in (("m512", (512, 512), 21), ("m256", (256, 256), 22), ("m300x400", (300, 400), 23), ("m640x600", (640, 600), 24)):
        img = torch.rand(1, 3, h, w, generator=torch.Generator().manual_seed(seed))
        with torch.no_grad():
            matte = ref_infer.InferenceWrapper.get_mask(fake_self, img)
        out[name] = {"seed": seed, "shape": (h, w), "matte_s4": matte[:, :, ::4, ::4].clone()}
    torch.save(out, GOLD / "masks.pt")
    print({k: (v["shape"], v.get("masks_sum")) for k, v in out.items()})
    print("bytes", (GOLD / "masks.pt").stat().st_size)


if __name__ == "__main__":
    main()
