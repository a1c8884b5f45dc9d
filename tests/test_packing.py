"""CPU: weight packing / BN folding / sub-pixel phase decomposition against torch's own operators,
and the drop-in modules' state_dict schema against the reference's."""
import json
import os

import numpy as np
import torch
import torch.nn.functional as F

from conftest import load_golden
from lama_b200 import _lib as L
from lama_b200 import modules as M
from lama_b200 import packing as P
from lama_b200.testing import BIG_LAMA_KWARGS, seeded_parameters_

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_conv_transpose_phases_equal_torch():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 8, 5, 7, generator=g, dtype=torch.float64)
    ct = torch.nn.ConvTranspose2d(8, 12, 3, stride=2, padding=1, output_padding=1).double()
    bn = torch.nn.BatchNorm2d(12).double()
    seeded_parameters_(bn, 1); seeded_parameters_(ct, 2, gain=1.0)
    bn.eval()
    want = torch.relu(bn(ct(x)))
    sc, sh = P.bn_scale_shift(bn)
    got = torch.zeros(2, 10, 14, 12, dtype=torch.float64)
    for a, b, pk in P.pack_conv_transpose_phases(ct.weight, ct.bias, sc, sh, act=L.ACT_RELU):
        got[:, a::2, b::2] = P.apply_packed_reference(pk, [x.permute(0, 2, 3, 1), None], (5, 7))
    np.testing.assert_allclose(got.permute(0, 3, 1, 2).detach().numpy(), want.detach().numpy(), atol=2e-6)


def test_pack_conv_reflect_stride2_equals_torch():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 8, 10, 12, generator=g, dtype=torch.float64)
    conv = torch.nn.Conv2d(8, 16, 3, stride=2, padding=1, padding_mode="reflect", bias=False).double()
    bn = seeded_parameters_(torch.nn.BatchNorm2d(16).double(), 3).eval()
    want = torch.relu(bn(conv(x)))
    sc, sh = P.bn_scale_shift(bn)
    pk = P.pack_conv([(conv.weight, 0, 0, 1)], sc, sh, stride=2, act=L.ACT_RELU)
    got = P.apply_packed_reference(pk, [x.permute(0, 2, 3, 1), None], (5, 6))
    np.testing.assert_allclose(got.permute(0, 3, 1, 2).detach().numpy(), want.detach().numpy(), atol=2e-6)


def test_split_bf16_precision():
    x = torch.randn(10000, generator=torch.Generator().manual_seed(2)) * 37.0
    s = P.split_bf16(x)
    rec = s[0].float() + s[1].float()
    assert float(((rec - x).abs() / x.abs().clamp_min(1e-30)).max()) <= 2.0 ** -16


def test_state_dict_schema_matches_reference():
    """989 generator entries for big-lama (SURVEY.md Appendix B); load_checkpoint uses strict=False, so
    key/shape drift would be silent — compare against the reference class when its tree is present,
    and always against the committed schema."""
    g = M.FFCResNetGenerator(**BIG_LAMA_KWARGS)
    ours = {k: tuple(v.shape) for k, v in g.state_dict().items()}
    assert len(ours) == 989
    schema_path = os.path.join(ROOT, "tests", "golden", "big_lama_state_dict_schema.json")
    from oracle import ref_import
    if ref_import.available():
        ref = ref_import.load_reference_ffc().FFCResNetGenerator(**BIG_LAMA_KWARGS)
        theirs = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
        assert ours == theirs
        ref.load_state_dict(g.state_dict(), strict=True)
        g.load_state_dict(ref.state_dict(), strict=True)
        if not os.path.isfile(schema_path):
            with open(schema_path, "w") as fh:
                json.dump({k: list(v) for k, v in theirs.items()}, fh)
    with open(schema_path) as fh:
        committed = {k: tuple(v) for k, v in json.load(fh).items()}
    assert ours == committed
    assert g.model[5].conv1.ffc.global_in_num == 384        # read by ffc.py:279 / refinement
    assert isinstance(g.model, torch.nn.Sequential) and len(g.model) == 36


def _seeded_like_reference(module, seed, golden):
    """seeded_parameters_(module, seed), checked to give the drop-in exactly the reference's state_dict: the same keys
    and shapes (what a strict load_state_dict checks) and, key by key, the same values (per-tensor sums of the
    reference module seeded alike, stored by tests/golden/make_golden.py)."""
    seeded_parameters_(module, seed)
    sd = module.state_dict()
    schema = json.loads(str(golden["sd_schema"]))
    assert {k: list(v.shape) for k, v in sd.items()} == schema
    np.testing.assert_allclose([sd[k].double().sum().item() for k in schema], golden["sd_sums"], rtol=1e-9, atol=1e-12)
    return module


def test_module_torch_composition_matches_reference_on_cpu():
    """Feature-fallback path (CPU tensors / unsupported options) is the reference's operator sequence: the reference
    FFC_BN_ACT's outputs on the same weights and inputs are stored in the golden."""
    a, _ = load_golden("surface_ffcbnact_32_k3_lfu_8x8")
    kw = dict(in_channels=32, out_channels=32, kernel_size=3, ratio_gin=0.75, ratio_gout=0.75, padding=1,
              activation_layer=torch.nn.ReLU, enable_lfu=True)
    ours = _seeded_like_reference(M.FFC_BN_ACT(**kw).eval(), 5, a)
    with torch.no_grad():
        c, d = ours((torch.from_numpy(a["x_l"]), torch.from_numpy(a["x_g"])))
    assert torch.allclose(torch.from_numpy(a["y_l"]), c, atol=1e-6)
    assert torch.allclose(torch.from_numpy(a["y_g"]), d, atol=1e-6)


def test_discriminator_surface_matches_reference():
    """FFCNLayerDiscriminator (ffc.py:370-433, training only) keeps the reference's state_dict and outputs (the
    reference's output and intermediate features on the same weights and input are stored in the golden)."""
    a, _ = load_golden("surface_discriminator_ndf16_32x32")
    kw = dict(input_nc=3, ndf=16, n_layers=3, init_conv_kwargs=dict(ratio_gin=0, ratio_gout=0.5, enable_lfu=False),
              conv_kwargs=dict(ratio_gin=0.5, ratio_gout=0.5, enable_lfu=False))
    ours = _seeded_like_reference(M.FFCNLayerDiscriminator(**kw).eval(), 9, a)
    fa = [torch.from_numpy(a[k]) for k in sorted(k for k in a if k.startswith("feat"))]
    with torch.no_grad():
        b, fb = ours(torch.from_numpy(a["x"]))
    assert torch.allclose(torch.from_numpy(a["y"]), b, atol=1e-6) and len(fa) == len(fb)
    assert all(torch.allclose(p, q, atol=1e-6) for p, q in zip(fa, fb))


# ------------------------------------------------------------------ property tests of the ffcb_conv contract
from hypothesis import given, settings, strategies as st  # noqa: E402


@settings(max_examples=25, deadline=None)
@given(k=st.sampled_from([1, 3]), stride=st.sampled_from([1, 2]), cin=st.sampled_from([4, 8, 12]),
       cout=st.sampled_from([4, 8]), h=st.integers(4, 11), w=st.integers(4, 11), seed=st.integers(0, 10 ** 6),
       reflect=st.booleans(), act=st.sampled_from([L.ACT_NONE, L.ACT_RELU, L.ACT_SIGMOID]))
def test_packed_conv_equals_torch_conv(k, stride, cin, cout, h, w, seed, reflect, act):
    """pack_conv + apply_packed_reference (the executable spec of ffcb_conv) == nn.Conv2d semantics for every
    kernel size / stride / border mode / ragged size the path uses."""
    g = torch.Generator().manual_seed(seed)
    pad = k // 2
    x = torch.randn(2, cin, h, w, generator=g, dtype=torch.float64)
    wt = torch.randn(cout, cin, k, k, generator=g, dtype=torch.float64)
    scale = torch.rand(cout, generator=g, dtype=torch.float64) + 0.5
    shift = torch.randn(cout, generator=g, dtype=torch.float64)
    xp = F.pad(x, (pad,) * 4, mode="reflect") if (reflect and pad) else F.pad(x, (pad,) * 4)
    want = F.conv2d(xp, wt, stride=stride) * scale[None, :, None, None] + shift[None, :, None, None]
    want = {L.ACT_NONE: want, L.ACT_RELU: want.clamp_min(0), L.ACT_SIGMOID: torch.sigmoid(want)}[act]
    pk = P.pack_conv([(wt, 0, 0, pad)], scale, shift, stride=stride,
                     border=L.BORDER_REFLECT if reflect else L.BORDER_ZERO, act=act)
    got = P.apply_packed_reference(pk, [x.permute(0, 2, 3, 1), None], tuple(want.shape[2:]))
    np.testing.assert_allclose(got.permute(0, 3, 1, 2).numpy(), want.numpy(), atol=2e-6)


def test_windowed_stem_packing_equals_reflect_conv7():
    """pack_stem_windowed over the packed NHWC8 image (ffcb_stem_pack layout) == ReflectionPad2d(3)+Conv2d(k7)+BN+ReLU."""
    g = torch.Generator().manual_seed(3)
    x = torch.rand(2, 4, 9, 13, generator=g, dtype=torch.float64)
    conv = torch.nn.Conv2d(4, 8, 7, bias=False).double()
    bn = seeded_parameters_(torch.nn.BatchNorm2d(8).double(), 4).eval()
    want = torch.relu(bn(conv(F.pad(x, (3, 3, 3, 3), mode="reflect"))))
    sc, sh = P.bn_scale_shift(bn)
    pk = P.pack_stem_windowed(conv.weight, sc, sh)
    packed = F.pad(F.pad(x, (3, 3, 3, 3), mode="reflect"), (0, 2, 0, 0, 0, 4)).permute(0, 2, 3, 1)   # [B,H+6,W+8,8]
    packed = packed.clone()
    packed[:, :-1, :, 4:8] = packed[:, 1:, :, 0:4]          # two-row packing of ffcb_stem_pack (Cin <= 4)
    assert len(pk.segs) == 4 and [s.dy for s in pk.segs] == [0, 2, 4, 6]
    wout = x.shape[3]
    window = torch.cat([packed[:, :, j:j + wout] for j in range(8)], dim=-1)                        # [B,H+6,W,64]
    got = P.apply_packed_reference(pk, [window, None], (x.shape[2], wout))
    np.testing.assert_allclose(got.permute(0, 3, 1, 2).detach().numpy(), want.detach().numpy(), atol=2e-6)


def test_windowed_stem_packing_with_more_than_four_input_channels():
    """Cin in 5..8 keeps one K-segment per kernel row (no room for a second row in the 8-channel pixel)."""
    g = torch.Generator().manual_seed(4)
    x = torch.rand(1, 6, 8, 10, generator=g, dtype=torch.float64)
    conv = torch.nn.Conv2d(6, 8, 7, bias=False).double()
    want = torch.relu(conv(F.pad(x, (3, 3, 3, 3), mode="reflect")))
    pk = P.pack_stem_windowed(conv.weight, torch.ones(8, dtype=torch.float64), torch.zeros(8, dtype=torch.float64))
    assert len(pk.segs) == 7
    packed = F.pad(F.pad(x, (3, 3, 3, 3), mode="reflect"), (0, 2, 0, 0, 0, 2)).permute(0, 2, 3, 1)
    window = torch.cat([packed[:, :, j:j + 10] for j in range(8)], dim=-1)
    got = P.apply_packed_reference(pk, [window, None], (8, 10))
    np.testing.assert_allclose(got.permute(0, 3, 1, 2).detach().numpy(), want.detach().numpy(), atol=2e-6)


def test_head_rows_plus_gather_equals_reflect_conv7():
    """pack_head_rows (kernel-row contraction) + the gather of ffcb_head_gather7 == ReflectionPad2d(3)+Conv2d(k7,bias)."""
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 8, 10, 12, generator=g, dtype=torch.float64)
    conv = torch.nn.Conv2d(8, 3, 7, bias=True).double()
    want = conv(F.pad(x, (3, 3, 3, 3), mode="reflect"))
    pk = P.pack_head_rows(conv.weight)
    q = P.apply_packed_reference(pk, [x.permute(0, 2, 3, 1), None], (10, 12))              # [B,H,W,24]
    w = 12
    xi = torch.arange(w)[:, None] + torch.arange(7)[None, :] - 3
    xi = xi.abs(); xi = torch.where(xi >= w, 2 * w - 2 - xi, xi)
    got = torch.stack([sum(q[:, :, xi[:, kx], n * 7 + kx] for kx in range(7)) + conv.bias[n] for n in range(3)], dim=1)
    np.testing.assert_allclose(got.detach().numpy(), want.detach().numpy(), atol=2e-6)
