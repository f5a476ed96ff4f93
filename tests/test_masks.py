"""Mask pre/post-processing around the external mask networks (SURVEY §8f rank 3).

CPU: the oracle restatement (oracle/restatement.py face_parsing_forward / modnet_get_mask) is pinned against outputs of the
UNMODIFIED reference code (face_parcing.py:55-81, notebooks/infer.py:649-684) recorded by oracle/make_golden_masks.py with the
seeded stand-in networks of oracle/stub_nets.py.  GPU: the device path (emoportraits_b200/masks.py over csrc/masks.cu) against
the same fixtures and, kernel by kernel, against torch on the same inputs."""
import pathlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

GOLD = pathlib.Path(__file__).parent / "golden" / "masks.pt"
PARSE = ("p512", "p256", "p300x400")
MATTE = ("m512", "m256", "m300x400", "m640x600")


def _gold():
    return torch.load(GOLD, weights_only=False)


def _unpack(packed, shape):
    n = int(np.prod(shape))
    return torch.from_numpy(np.unpackbits(np.asarray(packed))[:n].reshape(shape).astype(np.int64))


def _parsing_input(h, w, seed):
    from oracle.make_golden_masks import parsing_input

    return parsing_input(h, w, seed)


@pytest.mark.parametrize("name", PARSE)
def test_oracle_face_parsing_matches_reference(name):
    from oracle import restatement as R
    from oracle.stub_nets import StubBiSeNet

    g = _gold()[name]
    h, w = g["shape"]
    x = _parsing_input(h, w, g["seed"])
    with torch.no_grad():
        masks, y, labels = R.face_parsing_forward(StubBiSeNet(), x)
    assert torch.allclose(F.interpolate(((x - torch.tensor(R.PARSING_MEAN)[None, :, None, None]) / torch.tensor(R.PARSING_STD)[None, :, None, None]),
                                        size=(512, 512), mode="bilinear")[:, :, ::16, ::16], g["x512_s16"], atol=1e-6)
    for m, packed, total in zip(masks, g["masks_packed"], g["masks_sum"]):
        ref = _unpack(packed, m.shape)
        assert int(ref.sum()) == total
        assert m.dtype == torch.int64 and torch.equal(m, ref)


@pytest.mark.parametrize("name", MATTE)
def test_oracle_get_mask_matches_reference(name):
    from oracle import restatement as R
    from oracle.stub_nets import StubMODNet

    g = _gold()[name]
    h, w = g["shape"]
    img = torch.rand(1, 3, h, w, generator=torch.Generator().manual_seed(g["seed"]))
    with torch.no_grad():
        matte = R.modnet_get_mask(StubMODNet(), img)
    assert matte.shape == (1, 1, h, w)
    assert torch.allclose(matte[:, :, ::4, ::4], g["matte_s4"], atol=1e-6)


def test_face_parsing_rejects_mask_types_like_the_reference():
    from emoportraits_b200.masks import FaceParsing

    with pytest.raises(AttributeError):  # the reference's forward() raises AttributeError for every mask_type but None
        FaceParsing("face_hair", device="cpu", net=lambda x: (x,))


# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(512, 512), (256, 256), (300, 400), (700, 520), (1, 1)])
def test_parsing_prepare_kernel(hw):
    from emoportraits_b200 import masks, ops

    x = torch.rand(2, 3, *hw, generator=torch.Generator().manual_seed(3))
    mean, std = torch.tensor(masks.PARSING_MEAN), torch.tensor(masks.PARSING_STD)
    ref = F.interpolate((x - mean[None, :, None, None]) / std[None, :, None, None], size=(512, 512), mode="bilinear")
    got = ops.parsing_prepare(x.cuda(), mean.cuda(), std.cuda(), (512, 512)).cpu()
    assert (got - ref).abs().max().item() <= 2e-6  # the same taps and weights; sums may differ in the last bit


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(512, 512), (256, 256), (300, 400), (1024, 768)])
def test_parsing_masks_kernel(hw):
    from emoportraits_b200 import masks, ops
    from oracle import restatement as R

    y = torch.randn(2, 19, 512, 512, generator=torch.Generator().manual_seed(5))
    up = F.interpolate(y, size=hw, mode="bilinear")
    labels = up.argmax(1, keepdim=True)
    # pixels whose two best classes are closer than the interpolation rounding may legitimately flip
    top2 = up.topk(2, dim=1).values
    safe = (top2[:, :1] - top2[:, 1:2]) > 1e-5
    got, lab = ops.parsing_masks(y.cuda(), hw, R.parsing_label_sets(None), want_labels=True)
    assert torch.equal(lab.cpu().long()[safe], labels[safe])
    assert (~safe).float().mean().item() < 1e-3
    for k, labs in enumerate(R.parsing_label_sets(None)):
        ref = torch.zeros_like(labels)
        for i in labs:
            ref += labels == i
        assert torch.equal(got[k].cpu().long()[safe], ref[safe])


@pytest.mark.gpu
@pytest.mark.parametrize("io", [((512, 512), (512, 512)), ((256, 256), (512, 512)), ((512, 512), (256, 256)), ((300, 400), (512, 672)),
                                ((512, 672), (300, 400)), ((640, 600), (512, 480)), ((7, 5), (3, 11))])
def test_resize_area_kernel(io):
    from emoportraits_b200 import ops

    (hi, wi), (ho, wo) = io
    x = torch.rand(2, 3, hi, wi, generator=torch.Generator().manual_seed(7))
    ref = F.interpolate((x - 0.5) / 0.5, size=(ho, wo), mode="area")
    got = ops.resize_area(x.cuda(), (ho, wo), scale=2.0, shift=-1.0).cpu()
    assert (got - ref).abs().max().item() <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("name", PARSE)
def test_face_parsing_matches_reference_fixture(name):
    from emoportraits_b200.masks import FaceParsing
    from oracle.stub_nets import StubBiSeNet

    g = _gold()[name]
    h, w = g["shape"]
    x = _parsing_input(h, w, g["seed"])
    fp = FaceParsing(None, device="cuda", net=StubBiSeNet().cuda())
    masks = fp.forward(x.cuda())
    for m, packed in zip(masks, g["masks_packed"]):
        ref = _unpack(packed, m.shape)
        assert m.dtype == torch.int64 and m.shape == ref.shape
        # the stand-in network itself runs in torch on the GPU (its bicubic / conv kernels round differently from the CPU's, ~1e-4 on
        # the logits): labels may flip only where the two best classes tie to that level - a few pixels in ten thousand
        assert (m.cpu() != ref).float().mean().item() < 2e-3


@pytest.mark.gpu
@pytest.mark.parametrize("name", MATTE)
def test_get_mask_matches_reference_fixture(name):
    from emoportraits_b200.masks import modnet_get_mask
    from oracle.stub_nets import StubMODNet

    g = _gold()[name]
    h, w = g["shape"]
    img = torch.rand(1, 3, h, w, generator=torch.Generator().manual_seed(g["seed"]))
    matte = modnet_get_mask(StubMODNet().cuda(), img.cuda())
    assert matte.shape == (1, 1, h, w)
    # the stand-in network runs in torch on the GPU (rounds differently from the CPU run of the fixture); the two area resizes
    # around it are checked exactly in test_resize_area_kernel
    assert (matte.cpu()[:, :, ::4, ::4] - g["matte_s4"]).abs().max().item() <= 2e-4


@pytest.mark.gpu
def test_wrapper_uses_plugged_in_mask_networks():
    """InferenceWrapper.forward with face_idt / modnet plugged in follows notebooks/infer.py:408-426: the face mask multiplies the
    source image, the MODNet matte (computed on the unmasked crop) replaces the source mask when modnet_mask=True."""
    from emoportraits_b200.checkpoint import synthetic_head_pose_state_dict, synthetic_state_dict
    from emoportraits_b200.config import shipped_config
    from emoportraits_b200.infer import InferenceWrapper
    from emoportraits_b200.masks import FaceParsing, modnet_get_mask
    from oracle import frames as FR
    from oracle.stub_nets import StubBiSeNet, StubMODNet
    import tempfile

    size = 256
    cfg = shipped_config(size)
    golden = pathlib.Path(__file__).parent / "golden"
    with tempfile.TemporaryDirectory() as td:
        exp = pathlib.Path(td) / "logs" / "exp"
        exp.mkdir(parents=True)
        (exp / "args.txt").write_text((golden / f"args_{size}.txt").read_text())
        w = InferenceWrapper("exp", project_dir=td, folder="logs", state_dict=synthetic_state_dict(cfg, 0),
                             head_pose_state_dict=synthetic_head_pose_state_dict(0), print_params=False)
    src = FR.frame(size, 41, "smooth").cuda()
    with pytest.raises(NotImplementedError):
        w.forward(src, None, crop=False, modnet_mask=True)
    w.forward(src, None, crop=False)
    base_idt = w.idt_embed.clone()
    assert torch.equal(w.source_img_mask, torch.ones_like(src[:, :1]))
    w.face_idt = FaceParsing(None, device="cuda", net=StubBiSeNet().cuda())
    w.modnet = StubMODNet().cuda()
    w.forward(src, None, crop=False)
    fm = (w.face_idt.forward(src)[0] > 0.6).float()
    assert torch.equal(w.source_img_mask, fm) and torch.equal(w.source_img, src * fm)
    assert not torch.equal(w.idt_embed, base_idt)
    w.forward(src, None, crop=False, modnet_mask=True)
    assert torch.equal(w.source_img_mask, modnet_get_mask(w.modnet, src))
