"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

For each case the reference module (``saicinpainting/training/modules/ffc.py``, loaded by
``oracle/ref_import.py``) is constructed, its parameters are overwritten by the seeded
factory ``lama_b200.testing.seeded_parameters_``, it is run in ``eval()`` under
``no_grad`` on CPU fp32, and input / state_dict / output are stored in one ``.npz``.
The fixtures pin (a) the numpy and torch-CPU restatements in ``oracle/`` and (b), on the
GPU box where the reference tree is absent, the CUDA path itself.

Sizes are small on purpose (the whole directory stays < 4 MB).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.ref_import import load_reference_ffc  # noqa: E402
from lama_b200.testing import (seeded_parameters_, small_lama_kwargs, synthetic_image_mask,  # noqa: E402
                               generator_input)


def _sd_np(module):
    return {"sd::" + k: v.detach().cpu().numpy() for k, v in module.state_dict().items()
            if not k.endswith("num_batches_tracked")}


def _save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{name:32s} {os.path.getsize(path) / 1024:8.1f} KiB")


def _randn(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


@torch.no_grad()
def main():
    ffc = load_reference_ffc()
    torch.set_num_threads(1)

    # ---- FourierUnit: power-of-two, rectangular, odd and non-power-of-two planes
    fu_cases = {
        "fu_c8_16x16": (2, 8, 8, 16, 16),
        "fu_c4to6_8x32": (1, 4, 6, 8, 32),
        "fu_c16_32x32": (1, 16, 16, 32, 32),
        "fu_c4_15x15": (1, 4, 4, 15, 15),      # bin/to_jit.py traces at 120x120 -> 15x15 bottleneck
        "fu_c4_6x9": (2, 4, 4, 6, 9),          # odd width: no Nyquist column
        "fu_c2_20x24": (1, 2, 2, 20, 24),      # 2^a 3^b 5^c sizes (pad_out_to_modulo: 8 images)
    }
    for i, (name, (b, ci, co, h, w)) in enumerate(fu_cases.items()):
        m = seeded_parameters_(ffc.FourierUnit(ci, co).eval(), seed=10 + i, gain=1.0)
        x = _randn((b, ci, h, w), 100 + i)
        _save(name, x=x.numpy(), y=m(x).numpy(), **_sd_np(m))

    # ---- SpectralTransform (stride 1 no LFU = big-lama; stride 2; LFU on)
    st_cases = {
        "st_16to24_8x8": dict(ci=16, co=24, stride=1, lfu=False, hw=(8, 8)),
        "st_16to16_s2_16x16": dict(ci=16, co=16, stride=2, lfu=False, hw=(16, 16)),
        "st_16to16_lfu_8x8": dict(ci=16, co=16, stride=1, lfu=True, hw=(8, 8)),
    }
    for i, (name, c) in enumerate(st_cases.items()):
        m = seeded_parameters_(ffc.SpectralTransform(c["ci"], c["co"], stride=c["stride"],
                                                     enable_lfu=c["lfu"]).eval(), seed=20 + i, gain=1.0)
        x = _randn((2, c["ci"]) + c["hw"], 200 + i)
        _save(name, x=x.numpy(), y=m(x).numpy(), **_sd_np(m))

    # ---- FFC_BN_ACT: resblock flavour (0.75 / 0.75), stem flavour (local only, k7),
    #      downsample flavour (stride 2, local -> local+global)
    def run_ffc(name, seed, ctor_kw, xl_shape, xg_shape):
        m = seeded_parameters_(ffc.FFC_BN_ACT(**ctor_kw).eval(), seed=seed, gain=1.0)
        xl = _randn(xl_shape, seed + 300)
        xg = _randn(xg_shape, seed + 301) if xg_shape else 0
        yl, yg = m((xl, xg) if xg_shape else xl)
        arrays = dict(x_l=xl.numpy(), y_l=yl.numpy())
        if xg_shape:
            arrays["x_g"] = xg.numpy()
        if torch.is_tensor(yg):
            arrays["y_g"] = yg.numpy()
        _save(name, **arrays, **_sd_np(m))

    relu = torch.nn.ReLU
    run_ffc("ffcbnact_32_k3_075", 30,
            dict(in_channels=32, out_channels=32, kernel_size=3, ratio_gin=0.75, ratio_gout=0.75, padding=1,
                 activation_layer=relu, enable_lfu=False), (2, 8, 8, 8), (2, 24, 8, 8))
    run_ffc("ffcbnact_4to8_k7_local", 31,
            dict(in_channels=4, out_channels=8, kernel_size=7, ratio_gin=0, ratio_gout=0, padding=0,
                 activation_layer=relu, enable_lfu=False), (1, 4, 22, 22), None)
    run_ffc("ffcbnact_16to32_s2_to_global", 32,
            dict(in_channels=16, out_channels=32, kernel_size=3, ratio_gin=0, ratio_gout=0.75, stride=2,
                 padding=1, activation_layer=relu, enable_lfu=False), (2, 16, 16, 16), None)

    # ---- FFCResnetBlock (big-lama flavour, 32 channels)
    m = seeded_parameters_(
        ffc.FFCResnetBlock(32, padding_type="reflect", norm_layer=torch.nn.BatchNorm2d, activation_layer=relu,
                           ratio_gin=0.75, ratio_gout=0.75, enable_lfu=False).eval(), seed=40)
    xl, xg = _randn((2, 8, 16, 16), 400), _randn((2, 24, 16, 16), 401)
    yl, yg = m((xl, xg))
    _save("resblock_32_16x16", x_l=xl.numpy(), x_g=xg.numpy(), y_l=yl.numpy(), y_g=yg.numpy(), **_sd_np(m))

    # ---- small generator with the big-lama topology (ngf 8 -> 16+48 bottleneck channels, 2 blocks)
    kw = small_lama_kwargs(ngf=8, n_blocks=2)
    g = seeded_parameters_(ffc.FFCResNetGenerator(**kw).eval(), seed=50, gain=1.0)
    img, mask = synthetic_image_mask(2, 64, seed=5)
    x = generator_input(img, mask)
    _save("generator_ngf8_b2_64x64", image=img.numpy(), mask=mask.numpy(), x=x.numpy(), y=g(x).numpy(), **_sd_np(g))
    # rectangular, not a multiple of 64: 40 x 72 image -> 5 x 9 bottleneck
    img, mask = synthetic_image_mask(1, 40, seed=6, width=72)
    x = generator_input(img, mask)
    # same weights as generator_ngf8_b2_64x64 (state_dict stored there only)
    _save("generator_ngf8_b2_40x72", x=x.numpy(), y=g(x).numpy())


@torch.no_grad()
def make_predict():
    """Predict path (SURVEY.md row f1): PNG files -> reference InpaintingDataset -> reference generator -> bytes.

    The dataset / padding / decode code is the reference's own (saicinpainting/evaluation/data.py, imported from
    its file); DefaultInpaintingTrainingModule.forward and bin/predict.py need pytorch_lightning / hydra to import,
    so the six lines of theirs on this path are restated below with their file:line."""
    import importlib.util
    import tempfile
    from PIL import Image
    spec = importlib.util.spec_from_file_location(
        "_ref_eval_data", os.path.join(os.environ.get("LAMA_REFERENCE_ROOT", "/root/reference"),
                                       "saicinpainting/evaluation/data.py"))
    data = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(data)
    ffc = load_reference_ffc()
    torch.set_num_threads(1)
    g = seeded_parameters_(ffc.FFCResNetGenerator(**small_lama_kwargs(ngf=8, n_blocks=2)).eval(), seed=50, gain=1.0)

    rng = np.random.default_rng(7)
    b, h0, w0 = 3, 45, 52
    images = rng.integers(0, 256, size=(b, h0, w0, 3), dtype=np.uint8)
    images[0, :, :, :] = (np.linspace(0, 255, w0)[None, :, None] + np.zeros((h0, 1, 3))).astype(np.uint8)  # ramp
    masks = np.zeros((b, h0, w0), dtype=np.uint8)
    masks[0, 10:30, 12:40] = 255
    masks[1, 30:, 35:] = 255                 # touches the symmetric padding
    masks[1, 5:9, 5:9] = 1                   # "mask > 0" binarisation (predict.py:83)
    masks[2, ::7, ::5] = 128
    with tempfile.TemporaryDirectory() as d:
        for i in range(b):
            Image.fromarray(images[i]).save(os.path.join(d, f"im{i}.png"))
            Image.fromarray(masks[i]).save(os.path.join(d, f"im{i}_mask.png"))
        ds = data.InpaintingDataset(d, img_suffix=".png", pad_out_to_modulo=8)       # default.yaml:8-11
        items = [ds[i] for i in range(len(ds))]
    batch = {"image": torch.from_numpy(np.stack([it["image"] for it in items])),
             "mask": torch.from_numpy(np.stack([it["mask"] for it in items]))}
    unpad = items[0]["unpad_to_size"]
    batch["mask"] = (batch["mask"] > 0) * 1                                         # bin/predict.py:83
    img, mask = batch["image"], batch["mask"]
    masked_img = img * (1 - mask)                                                   # trainers/default.py:59
    masked_img = torch.cat([masked_img, mask], dim=1)                               # trainers/default.py:68
    predicted = g(masked_img)                                                       # trainers/default.py:70
    inpainted = mask * predicted + (1 - mask) * img                                 # trainers/default.py:71
    outs = []
    for i in range(b):
        cur = inpainted[i].permute(1, 2, 0).numpy()                                 # bin/predict.py:85
        cur = cur[:unpad[0], :unpad[1]]                                             # bin/predict.py:88-91
        outs.append(np.clip(cur * 255, 0, 255).astype("uint8"))                     # bin/predict.py:93
    # weights: same as generator_ngf8_b2_64x64 (state_dict stored there only)
    _save("predict_ngf8_3x45x52", images=images, masks=masks, x=masked_img.numpy(), predicted=predicted.numpy(),
          out=np.stack(outs))


@torch.no_grad()
def make_f4():
    """Round 2, SURVEY.md row f4: optional FFC flags that became native — LFU (ffc.py:148-157) and the stride-2
    SpectralTransform (ffc.py:122-125), alone and inside an FFC_BN_ACT / FFCResnetBlock.  Channel counts large enough
    for the native views (LFU quadrants carry c/4 channels, every view needs a multiple of 4)."""
    ffc = load_reference_ffc()
    torch.set_num_threads(1)
    relu = torch.nn.ReLU
    st_cases = {
        "st_32to32_lfu_8x8": dict(ci=32, co=32, stride=1, lfu=True, hw=(8, 8)),
        "st_32to32_s2_lfu_16x16": dict(ci=32, co=32, stride=2, lfu=True, hw=(16, 16)),
        "st_32to64_s2_12x20": dict(ci=32, co=64, stride=2, lfu=False, hw=(12, 20)),
    }
    for i, (name, c) in enumerate(st_cases.items()):
        m = seeded_parameters_(ffc.SpectralTransform(c["ci"], c["co"], stride=c["stride"],
                                                     enable_lfu=c["lfu"]).eval(), seed=60 + i, gain=1.0)
        x = _randn((2, c["ci"]) + c["hw"], 600 + i)
        _save(name, x=x.numpy(), y=m(x).numpy(), **_sd_np(m))
    # FourierUnit with spectral_pos_encoding (ffc.py:91-95), alone and inside a SpectralTransform
    m = seeded_parameters_(ffc.FourierUnit(8, 8, spectral_pos_encoding=True).eval(), seed=65, gain=1.0)
    x = _randn((2, 8, 12, 16), 650)
    _save("fu_c8_pos_12x16", x=x.numpy(), y=m(x).numpy(), **_sd_np(m))
    m = seeded_parameters_(ffc.SpectralTransform(16, 32, enable_lfu=False, spectral_pos_encoding=True).eval(),
                           seed=66, gain=1.0)
    x = _randn((2, 16, 8, 8), 660)
    _save("st_16to32_pos_8x8", x=x.numpy(), y=m(x).numpy(), **_sd_np(m))
    # generator with out_ffc=True (ffc.py:356-358): an inline FFCResnetBlock at full resolution before the head
    kw = small_lama_kwargs(ngf=16, n_blocks=1, n_downsampling=2)
    kw.update(out_ffc=True, out_ffc_kwargs=dict(ratio_gin=0.5, ratio_gout=0.5, enable_lfu=False))
    g = seeded_parameters_(ffc.FFCResNetGenerator(**kw).eval(), seed=67, gain=1.0)
    img, mask = synthetic_image_mask(1, 32, seed=8)
    x = generator_input(img, mask)
    _save("generator_ngf16_outffc_32x32", x=x.numpy(), y=g(x).numpy(), **_sd_np(g))
    # FFC_BN_ACT with a global input AND stride 2 (the spectral branch pools, the 3x3 convs stride), LFU on
    m = seeded_parameters_(ffc.FFC_BN_ACT(in_channels=64, out_channels=64, kernel_size=3, ratio_gin=0.5, ratio_gout=0.5,
                                          stride=2, padding=1, activation_layer=relu, enable_lfu=True).eval(),
                           seed=70, gain=1.0)
    xl, xg = _randn((2, 32, 16, 16), 700), _randn((2, 32, 16, 16), 701)
    yl, yg = m((xl, xg))
    _save("ffcbnact_64_s2_lfu_16x16", x_l=xl.numpy(), x_g=xg.numpy(), y_l=yl.numpy(), y_g=yg.numpy(), **_sd_np(m))
    # residual block with LFU (the reference's default enable_lfu=True flavour, e.g. configs/training/lama-fourier)
    m = seeded_parameters_(
        ffc.FFCResnetBlock(64, padding_type="reflect", norm_layer=torch.nn.BatchNorm2d, activation_layer=relu,
                           ratio_gin=0.5, ratio_gout=0.5, enable_lfu=True).eval(), seed=71)
    xl, xg = _randn((1, 32, 8, 8), 710), _randn((1, 32, 8, 8), 711)
    yl, yg = m((xl, xg))
    _save("resblock_64_lfu_8x8", x_l=xl.numpy(), x_g=xg.numpy(), y_l=yl.numpy(), y_g=yg.numpy(), **_sd_np(m))


def _sd_fingerprint(module):
    """state_dict schema (every key, num_batches_tracked included, with its shape) and one float64 sum per tensor:
    enough to show that ``seeded_parameters_`` gives a drop-in module the reference's values under the same keys,
    without storing the weights."""
    import json
    sd = module.state_dict()
    return dict(sd_schema=np.asarray(json.dumps({k: list(v.shape) for k, v in sd.items()})),
                sd_sums=np.asarray([v.double().sum().item() for v in sd.values()]))


@torch.no_grad()
def make_surface():
    """Module surface kept identical to the reference beyond the generator: the FFC_BN_ACT torch composition with
    LFU (the CPU / unsupported-option path) and FFCNLayerDiscriminator (ffc.py:370-433, training only)."""
    ffc = load_reference_ffc()
    torch.set_num_threads(1)
    kw = dict(in_channels=32, out_channels=32, kernel_size=3, ratio_gin=0.75, ratio_gout=0.75, padding=1,
              activation_layer=torch.nn.ReLU, enable_lfu=True)
    m = seeded_parameters_(ffc.FFC_BN_ACT(**kw).eval(), 5)
    xl, xg = _randn((1, 8, 8, 8), 800), _randn((1, 24, 8, 8), 801)
    yl, yg = m((xl, xg))
    _save("surface_ffcbnact_32_k3_lfu_8x8", x_l=xl.numpy(), x_g=xg.numpy(), y_l=yl.numpy(), y_g=yg.numpy(),
          **_sd_fingerprint(m))
    kw = dict(input_nc=3, ndf=16, n_layers=3, init_conv_kwargs=dict(ratio_gin=0, ratio_gout=0.5, enable_lfu=False),
              conv_kwargs=dict(ratio_gin=0.5, ratio_gout=0.5, enable_lfu=False))
    m = seeded_parameters_(ffc.FFCNLayerDiscriminator(**kw).eval(), 9)
    x = _randn((1, 3, 32, 32), 1)
    y, feats = m(x)
    _save("surface_discriminator_ndf16_32x32", x=x.numpy(), y=y.numpy(),
          **{f"feat{i}": f.numpy() for i, f in enumerate(feats)}, **_sd_fingerprint(m))


if __name__ == "__main__":
    if "--f4-only" in sys.argv:
        make_f4()
    elif "--predict-only" in sys.argv:
        make_predict()
    elif "--surface-only" in sys.argv:
        make_surface()
    else:
        main()
        make_predict()
        make_f4()
        make_surface()
