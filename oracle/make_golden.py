"""TEST INFRASTRUCTURE ONLY.  Generates the golden fixtures under tests/golden/ by running the UNMODIFIED reference
(/root/reference, through oracle/ref_harness.py) in this container.  /root/reference cannot travel to the GPU box,
so the fixtures are committed together with this script:

    python -m oracle.make_golden            # writes tests/golden/*.pt and the checkpoint-layout manifests
    python -m oracle.make_golden options    # tests/golden/va256_options.pt: the non-default forward() arguments

What is recorded, for image_size 256 and 512 (shipped config, experiments/args.txt):
  * the checkpoint layout (key -> shape) of va.Model.state_dict() and of the head-pose resnet18;
  * the reference InferenceWrapper's outputs for seeded synthetic frames with the seeded synthetic checkpoint of
    emoportraits_b200.checkpoint.synthetic_state_dict (loaded with load_state_dict(strict=True) into the reference
    model, which is itself the proof that our structural layout spec equals the reference's):
    final image, pre-sigmoid logits, and stage-boundary taps (large tensors strided down to keep fixtures small).
"""
from __future__ import annotations

import pathlib
import sys

import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
GOLD = ROOT / "tests" / "golden"

SRC_SEED, DRV_SEEDS = 0, (1, 2)


def sub(t: torch.Tensor, max_elems: int = 20000, thin: int = 4):
    """deterministic strided subsample of a large tensor: returns (flat_values, stride).  The stride is `thin` times the one
    that keeps max_elems values (thin=4 keeps each stage-1 fixture file under 1 MB)."""
    f = t.detach().float().reshape(-1)
    stride = max(1, (f.numel() + max_elems - 1) // max_elems) * thin
    return f[::stride].clone(), stride


def run(image_size: int):
    import oracle.ref_harness as H
    from emoportraits_b200.checkpoint import (state_dict_spec, head_pose_spec, synthetic_state_dict,
                                              synthetic_head_pose_state_dict)
    from emoportraits_b200.config import shipped_config

    w, msd, hsd, lines = H.build_reference_wrapper(image_size, 0)
    cfg = shipped_config(image_size)

    # ---- layout manifests (from the REFERENCE objects) ----
    (GOLD / f"state_dict_manifest_{image_size}.txt").write_text(
        "".join(f"{k} {tuple(v.shape)}\n" for k, v in msd.items()))
    (GOLD / "head_pose_manifest.txt").write_text("".join(f"{k} {tuple(v.shape)}\n" for k, v in hsd.items()))
    (GOLD / f"args_{image_size}.txt").write_text("".join(lines))
    spec = state_dict_spec(cfg)
    assert {k: tuple(v.shape) for k, v in msd.items()} == {k: tuple(v) for k, v in spec.items()}, "layout spec mismatch"
    assert {k: tuple(v.shape) for k, v in hsd.items()} == {k: tuple(v) for k, v in head_pose_spec().items()}

    # ---- seeded synthetic checkpoint into the reference model ----
    sd = synthetic_state_dict(cfg, seed=0)
    hp = synthetic_head_pose_state_dict(seed=0)
    # aligned_keypoints is a buffer read from data/aligned_keypoints_3d.npy; keep the reference's own values
    sd["expression_embedder_nw.aligned_keypoints"] = msd["expression_embedder_nw.aligned_keypoints"]
    missing = w.model.load_state_dict(sd, strict=True)
    w.model.head_pose_regressor.net.load_state_dict(hp, strict=True)
    w.model.eval()
    w.model.head_pose_regressor.net.eval()

    taps = {}
    hooks = []
    hooks.append(w.model.decoder_nw.img_decoder.dec_img_head[2].register_forward_hook(
        lambda m, i, o: taps.__setitem__("logits", o.detach().clone())))
    hooks.append(w.model.uv_generator_nw.register_forward_hook(
        lambda m, i, o: taps.__setitem__("uv_warp", o[0].detach().clone())))
    hooks.append(w.model.decoder_nw.register_forward_pre_hook(
        lambda m, i: taps.__setitem__("aligned_feat2d", i[2].detach().clone())))
    hooks.append(w.model.decoder_nw.res_decoder.register_forward_hook(
        lambda m, i, o: taps.__setitem__("dec_feat", o.detach().clone())))

    from oracle import frames as FR
    from oracle import restatement as R

    out = {"image_size": image_size, "cases": []}
    for kind, src_seed, drv_seeds in (("noise", SRC_SEED, DRV_SEEDS), ("smooth", 10, (11, 12))):
        case = {"kind": kind, "src_seed": src_seed, "drv_seeds": list(drv_seeds), "frames": []}
        src = FR.pil(image_size, src_seed, kind)
        first = True
        for ds in drv_seeds:
            drv = FR.pil(image_size, ds, kind)
            with torch.no_grad():
                res = w.forward(src if first else None, drv, crop=False, mix=True, mix_old=False)
            if first:
                ths = w.pred_source_theta.clone()
                case["source"] = {
                    "idt_embed": w.idt_embed.clone(),
                    "pred_source_theta": ths,
                    # the reference's own fp32 pose algebra on THIS machine (torch CPU LU inverse; infer.py:443,
                    # expression_embedder.py:168): lets a test inject bit-identical pose matrices into the GPU path
                    "inv_warp": ths.float().inverse()[:, :3].clone(),
                    "align2d": R.align_theta_2d(ths[:, :3]).clone(),
                    "pred_source_pose_embed": w.pred_source_pose_embed.clone(),
                    "xy_warp": sub(w.source_xy_warp_resize),
                    "source_latent_volume": sub(w.source_latent_volume),
                    "target_latent_volume_1": sub(w.target_latent_volume_1),
                    "target_latent_volume": sub(w.target_latent_volume),
                }
                first = False
            case["frames"].append({
                "seed": ds,
                # strided subsamples keep the committed fixtures small (every 16th / 64th pixel value)
                "img": sub(res[1], 50000),
                "logits": sub(taps["logits"], 50000),
                "pred_target_theta": w.pred_target_theta.clone(),
                "align2d": R.align_theta_2d(w.pred_target_theta[:, :3]).clone(),
                "target_pose_embed": w.target_pose_embed.clone(),
                "uv_warp": sub(taps["uv_warp"]),
                "aligned_feat2d": sub(taps["aligned_feat2d"]),
                "dec_feat": sub(taps["dec_feat"]),
            })
            print(f"[golden {image_size} {kind}] frame seed {ds}: img mean {res[1].mean().item():.4f} "
                  f"logits [{taps['logits'].min().item():.2f}, {taps['logits'].max().item():.2f}]")
        out["cases"].append(case)
    for h in hooks:
        h.remove()
    torch.save(out, GOLD / f"va{image_size}_seed0.pt")
    return out


def run_stage2(output_size: int = 512, batch: int = 1):
    """Golden fixtures of the stage-2 refinement path: reference notebooks/infer_s2.py InferenceWrapper.forward with the
    seeded synthetic stage-2 checkpoint (load_state_dict strict), smooth synthetic frames at 256^2 resized up."""
    import oracle.ref_harness as H
    from emoportraits_b200.stage2 import Stage2Config, state_dict_spec_s2, synthetic_state_dict_s2
    from oracle import frames as FR

    w, msd, lines = H.build_reference_stage2(output_size, 0)
    cfg = Stage2Config(output_size=output_size)
    (GOLD / f"state_dict_manifest_s2_{output_size}.txt").write_text("".join(f"{k} {tuple(v.shape)}\n" for k, v in msd.items()))
    (GOLD / f"args_s2_{output_size}.txt").write_text("".join(lines))
    assert {k: tuple(v.shape) for k, v in msd.items()} == {k: tuple(v) for k, v in state_dict_spec_s2(cfg).items()}
    sd = synthetic_state_dict_s2(cfg, 0)
    w.model_two.load_state_dict(sd, strict=True)
    w.model_two.eval()
    taps = {}
    h = w.model_two.decoder.register_forward_hook(lambda m, i, o: taps.__setitem__("add", o[0].detach().clone()))
    h2 = w.model_two.local_encoder.register_forward_hook(lambda m, i, o: taps.__setitem__("vol", o.detach().clone()))
    seeds = list(range(50, 50 + batch))
    img = torch.cat([FR.frame(256, s, "smooth") for s in seeds])
    with torch.no_grad():
        pil, pil_resized, pil_ffhq, mask = w.forward(img)
    h.remove(); h2.remove()
    import numpy as np
    ffhq8 = np.stack([np.asarray(p) for p in pil_ffhq])
    out = {"output_size": output_size, "seeds": seeds, "input_size": 256, "vol": sub(taps["vol"], 40000, 1), "add": sub(taps["add"], 60000, 1),
           "ffhq_uint8": sub(torch.from_numpy(ffhq8.astype(np.float32)), 60000, 1)}
    print(f"[golden s2 {output_size} b{batch}] add range [{taps['add'].min().item():.3f}, {taps['add'].max().item():.3f}] vol max {taps['vol'].abs().max().item():.2f}")
    torch.save(out, GOLD / f"s2_{output_size}_b{batch}.pt")


# ------------------------------------------------------------------------------------------------------------------
# the non-default arguments of InferenceWrapper.forward (notebooks/infer.py:355-357) that change the hot path
# ------------------------------------------------------------------------------------------------------------------
OPT_SRC, OPT_DRV = 10, (11, 12, 13)


def option_inputs(image_size: int, cfg):
    """Seeded inputs of the option cases, shared by this generator and the tests (tests/test_forward_options*.py)."""
    g = torch.Generator().manual_seed(1234)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, image_size), torch.linspace(-1, 1, image_size), indexing="ij")
    r = (xx * xx + (yy * 1.1) ** 2).sqrt()
    mask = ((0.85 - r) / 0.2).clamp(0, 1)[None, None].contiguous()          # soft disc, exactly 0 near the corners
    return {
        "source_mask": mask,
        "driver_mask": (1 - mask).contiguous(),                               # must not change the result (use_seg=False)
        "pose_embed": (torch.randn(1, 128, generator=g) * 0.1),
        "theta_embed": (torch.tensor([[1.05, 0.95, 1.0]]), torch.tensor([[0.25, -0.12, 0.08]]),
                        torch.tensor([[0.04, 0.02, -0.03]])),
        "c_source_latent_volume": _smooth_volume(cfg, g),
        "c_target_latent_volume": _smooth_volume(cfg, g),
    }


def _smooth_volume(cfg, g):
    """band-limited (1,C,D,S,S) volume: one seeded plane wave per channel, amplitude 0.5 (a white-noise volume would make
    the trilinear warps differentiate rounding noise, like the white-noise frames of tests/test_oracle_golden.py)"""
    z, y, x = torch.meshgrid(torch.linspace(-1, 1, cfg.D), torch.linspace(-1, 1, cfg.S), torch.linspace(-1, 1, cfg.S), indexing="ij")
    k = (torch.rand(cfg.C, 3, generator=g) * 2 - 1) * 4.0
    ph = torch.rand(cfg.C, generator=g) * 6.2831853
    v = torch.sin(k[:, 0, None, None, None] * x + k[:, 1, None, None, None] * y + k[:, 2, None, None, None] * z + ph[:, None, None, None])
    return (0.5 * v)[None].contiguous()


def run_options(image_size: int = 256):
    """Runs the UNMODIFIED reference wrapper with each non-default forward() argument that reaches the hot path and
    records the image (strided) and the pose it used: mix_old=True, smooth_pose=True over three frames,
    custome_target_pose_embed, custome_target_theta_embed, source_mask (+ a driver_mask that must be ignored),
    target_theta=False, c_source_latent_volume, c_target_latent_volume, mix=False."""
    import oracle.ref_harness as H
    from emoportraits_b200.checkpoint import synthetic_head_pose_state_dict, synthetic_state_dict
    from emoportraits_b200.config import shipped_config
    from oracle import frames as FR

    w, msd, hsd, lines = H.build_reference_wrapper(image_size, 0)
    cfg = shipped_config(image_size)
    sd = synthetic_state_dict(cfg, seed=0)
    sd["expression_embedder_nw.aligned_keypoints"] = msd["expression_embedder_nw.aligned_keypoints"]
    w.model.load_state_dict(sd, strict=True)
    w.model.head_pose_regressor.net.load_state_dict(synthetic_head_pose_state_dict(seed=0), strict=True)
    w.model.eval()
    w.model.head_pose_regressor.net.eval()
    kind = "smooth"
    src = FR.pil(image_size, OPT_SRC, kind)
    drv = [FR.pil(image_size, s, kind) for s in OPT_DRV]
    X = option_inputs(image_size, cfg)
    base = dict(crop=False, mix=True, mix_old=False)
    out = {"image_size": image_size, "kind": kind, "src_seed": OPT_SRC, "drv_seeds": list(OPT_DRV), "cases": {}}

    def rec(name, res, **extra):
        d = {"img": sub(res[1], 50000), "pred_target_theta": w.pred_target_theta.clone(),
             "target_pose_embed": w.target_pose_embed.clone()}
        d.update(extra)
        out["cases"][name] = d
        print(f"[golden options {image_size}] {name}: img mean {res[1].mean().item():.4f}")

    with torch.no_grad():
        rec("default", w.forward(src, drv[0], **base))
        rec("mix_old", w.forward(src, drv[0], crop=False, mix=True, mix_old=True))
        rec("no_mix", w.forward(src, drv[0], crop=False, mix=False))
        rec("target_theta_false", w.forward(src, drv[0], target_theta=False, **base))
        # smooth_pose: self.theta starts at the first frame's pose and is smoothed over the next calls (pose_momentum 0.5)
        w.forward(src, None, **base)
        for i, d in enumerate(drv):
            rec(f"smooth_pose_{i}", w.forward(None, d, smooth_pose=True, reset_tracking=(i == 0), **base))
        rec("custome_target_pose_embed", w.forward(src, drv[0], custome_target_pose_embed=X["pose_embed"].clone(), **base))
        rec("custome_target_theta_embed", w.forward(src, drv[0], custome_target_theta_embed=tuple(t.clone() for t in X["theta_embed"]), **base))
        rec("source_mask", w.forward(src, drv[0], source_mask=X["source_mask"].clone(), driver_mask=X["driver_mask"].clone(), **base),
            idt_embed=w.idt_embed.clone(), pred_source_theta=w.pred_source_theta.clone())
        rec("c_source_latent_volume", w.forward(src, drv[0], c_source_latent_volume=X["c_source_latent_volume"].clone(), **base))
        rec("c_target_latent_volume", w.forward(src, drv[0], c_target_latent_volume=X["c_target_latent_volume"].clone(), **base))
    torch.save(out, GOLD / f"va{image_size}_options.pt")
    return out


if __name__ == "__main__":
    GOLD.mkdir(parents=True, exist_ok=True)
    if sys.argv[1:2] == ["options"]:
        run_options(int(sys.argv[2]) if len(sys.argv) > 2 else 256)
    elif sys.argv[1:2] == ["s2"]:
        run_stage2(int(sys.argv[2]) if len(sys.argv) > 2 else 512, int(sys.argv[3]) if len(sys.argv) > 3 else 1)
    else:
        sizes = [int(a) for a in sys.argv[1:]] or [256, 512]
        for s in sizes:
            run(s)


