"""Pipeline parity (SURVEY.md 8 rows a-15, a-16): ``VisualClozeModel.process_images`` / ``.upsampling`` against a composition of
oracle pieces (oracle/pipeline_oracle.py: reference-equivalent mask packing and cond concat, the UNMODIFIED reference
``prepare_modified``, sampler + model oracle, ``vae_oracle.decode``, query-row crop, SDEdit blend) on the same injected stub
encoders.  The composition needs the reference's own ``prepare_modified``, so its sampler inputs and final images were run once
on a B200 and stored in tests/golden/pipeline_small.pt (``python oracle/gen_golden_gpu.py``).

  packed ``img_cond``, ``img_ids``, noise tokens, ``txt`` / ``y`` / masks / guidance handed to the sampler   bit-exact
  final PIL images                                                                                           PSNR >= 35 dB
"""
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


def _psnr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    mse = ((a - b) ** 2).mean()
    return 10 * math.log10(255.0 ** 2 / max(mse, 1e-12))


@pytest.fixture(scope="module")
def rig():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return _rig()


@pytest.fixture(scope="module")
def golden():
    return torch.load(os.path.join(GOLDEN, "pipeline_small.pt"), weights_only=False)


def _rig():
    from oracle import flux_oracle as fo, vae_oracle as vo
    import visualcloze_b200.model as M
    from visualcloze_b200 import pipeline as P, vae as V
    g = torch.load(os.path.join(GOLDEN, "flux_small_b1.pt"), weights_only=False)
    cfg = fo.FluxConfig(**g["cfg"])
    params = {k: v.cuda() for k, v in fo.make_params(cfg, seed=g["param_seed"]).items()}
    fp = M.FluxParams(**{k: v for k, v in g["cfg"].items() if k not in ("lora_rank", "lora_scale")})
    with torch.device("cuda"):
        model = M.FluxLoraWrapper(lora_rank=cfg.lora_rank, params=fp)
    model.load_state_dict(params, strict=True)
    vsmall = dict(ch=64, ch_mult=[1, 2, 2, 2], num_res_blocks=1)
    dec = V.AutoEncoderDecoder(V.AutoEncoderParams(**vsmall), device="cuda").init_synthetic(1)
    vae_cfg = vo.VaeConfig(out_ch=3, z_channels=16, **vsmall)
    vae_p = {k: v.float() for k, v in dec.state_dict().items()}

    def t5(prompts):
        gg = torch.Generator().manual_seed(sum(map(len, prompts)))
        return (0.3 * torch.randn(len(prompts), 24, 64, generator=gg)).to(BF16).cuda()

    def clip(prompts):
        return torch.randn(len(prompts), 32, generator=torch.Generator().manual_seed(7)).to(BF16).cuda()

    def encode(x):                       # stands in for AutoencoderKL.encode(x).latent_dist.sample(): bf16 in, bf16 latent out
        gg = torch.Generator(device="cuda").manual_seed(int(x.shape[-1]) + int(x.float().abs().sum().item() * 7) % 1000)
        return torch.randn(x.shape[0], 16, x.shape[2] // 8, x.shape[3] // 8, generator=gg, device="cuda").to(BF16)

    pipe = P.VisualClozeModel(None, resolution=64, model=model, ae_decoder=dec, t5=t5, clip=clip, encode=encode)
    return dict(pipe=pipe, t5=t5, clip=clip, encode=encode, flux_p=params, flux_cfg=cfg, vae_p=vae_p, vae_cfg=vae_cfg)


def _spy_sampler(pipe, seen):
    """record what the pipeline hands to the sampler (x, model_kwargs) without changing it"""
    make = pipe._make_sample_fn

    def wrapped(*a, **k):
        fn = make(*a, **k)

        def spy(x, model, kw):
            seen.append(dict(kw, x=x))
            return fn(x, model, kw)
        return spy
    pipe._make_sample_fn = wrapped
    return make


def _grid():
    from PIL import Image
    rng = np.random.RandomState(0)
    mk = lambda: Image.fromarray(rng.randint(0, 255, (90, 90, 3), dtype=np.uint8))
    imgs = [[mk() for _ in range(3)] for _ in range(2)]
    imgs[1][2] = None
    return imgs


TAPS = ("x", "cond", "img_ids", "txt", "txt_ids", "txt_mask", "y", "img_mask", "guidance")


def _same_inputs(ours: dict, orc: dict):
    for k in TAPS:
        a, b = ours[k], orc[k]
        assert a.shape == b.shape and a.dtype == b.dtype, (k, a.shape, b.shape, a.dtype, b.dtype)
        assert torch.equal(a.cpu(), b.cpu()), f"{k}: packed sampler input differs from the reference composition"


def _oracle_kwargs(rig):
    return {k: rig[k] for k in ("t5", "clip", "encode", "flux_p", "flux_cfg", "vae_p", "vae_cfg")}


def oracle_process_images(rig):
    """The reference composition for test_process_images_matches_oracle_composition: (sampler inputs, [cropped result])."""
    from oracle import pipeline_oracle as po
    pipe = rig["pipe"]
    pipe.set_grid_size(2, 3)
    cells, mask_position, _ = pipe._prepare_grid([[im.convert("RGB") if im is not None else None for im in row] for row in _grid()])
    taps = {}
    ref, query, _ = po.process_images(cells, mask_position, 2, 3, ["layout prompt", "task prompt", "content prompt"], 5, 30, 4,
                                      device=torch.device("cuda"), taps=taps, **_oracle_kwargs(rig))
    return {k: taps[k].cpu() for k in TAPS}, [np.asarray(im) for im in ref]


def oracle_upsampling(rig):
    """The reference composition for test_upsampling_matches_oracle_composition: (sampler inputs, result)."""
    from PIL import Image
    from oracle import pipeline_oracle as po
    rng = np.random.RandomState(3)
    img = Image.fromarray(rng.randint(0, 255, (64, 64, 3), dtype=np.uint8))
    taps = {}
    g2 = torch.Generator(device="cuda").manual_seed(11)
    ref = po.upsampling(img, (80, 96), 30, 4, 0.4, g2, "a cat", device=torch.device("cuda"), taps=taps, **_oracle_kwargs(rig))
    return {k: taps[k].cpu() for k in TAPS}, np.asarray(ref)


def test_process_images_matches_oracle_composition(rig, golden):
    pipe = rig["pipe"]
    pipe.set_grid_size(2, 3)
    seen = []
    orig = _spy_sampler(pipe, seen)
    try:
        out = pipe.process_images(_grid(), ["layout prompt", "task prompt", "content prompt"], seed=5, cfg=30, steps=4, is_upsampling=False)
    finally:
        pipe._make_sample_fn = orig
    taps, ref = golden["process_images"]
    assert len(seen) == 1
    _same_inputs(seen[0], taps)
    assert len(out) == len(ref) == 1 and out[0].size == (64, 64) and ref[0].shape == (64, 64, 3)
    p = _psnr(out[0], ref[0])
    print(f"[pipeline] process_images PSNR vs oracle composition: {p:.1f} dB")
    assert p >= 35.0, f"PSNR {p:.1f} dB"


def test_upsampling_matches_oracle_composition(rig, golden):
    """SDEdit second stage: blend ``noise * (1 - s) + latent * s`` (visualcloze.py:221), all-ones mask over a blank condition,
    1x1 grid, do_shift=False schedule from ``strength``."""
    from PIL import Image
    pipe = rig["pipe"]
    rng = np.random.RandomState(3)
    img = Image.fromarray(rng.randint(0, 255, (64, 64, 3), dtype=np.uint8))
    seen = []
    orig = _spy_sampler(pipe, seen)
    try:
        g1 = torch.Generator(device="cuda").manual_seed(11)
        out = pipe.upsampling(img, (80, 96), 30, upsampling_steps=4, upsampling_noise=0.4, generator=g1,
                              content_prompt="The last image of the last row depicts: a cat")
    finally:
        pipe._make_sample_fn = orig
    taps, ref = golden["upsampling"]
    assert len(seen) == 1
    _same_inputs(seen[0], taps)
    assert out.size == (80, 96) and ref.shape == (96, 80, 3)
    p = _psnr(out, ref)
    print(f"[pipeline] upsampling PSNR vs oracle composition: {p:.1f} dB")
    assert p >= 35.0, f"PSNR {p:.1f} dB"
