"""CPU: E2VIDRecurrent with use_upsample_conv=False (TransposedConvLayer decoders, model/e2vid/unet.py).

* the polyphase packing: the packed 3x3 phase convolution, unpacked from the layer's K-major weights and followed by
  the phase shuffle, is ConvTranspose2d(5, stride 2, padding 2, output_padding 1);
* construction: the reference's key set and shapes, strict load, norm='BN' still refused;
* the tests' transposed decoder (e2vid_transposed_ref) against nn.ConvTranspose2d + ReLU run as a module, and its
  whole step against the oracle's upsample-conv step with the decoders swapped out;
* with the reference tree present: strict load into the reference model and its frames against e2vid_transposed_ref."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from bde2vid_b200 import synth
from bde2vid_b200.e2vid import E2VIDRecurrent, _TransposedConvLayer, _transposed_layer
from e2vid_transposed_ref import e2vid_transposed_forward, transposed_conv
from oracle import ref_shim


def unpack(layer, cin):
    """_Layer.w [4*Cout, Kpad] back to [4*Cout, Cin, 3, 3], for either K order of _pack_conv."""
    n = layer.w.shape[0]
    w = layer.w[:, :9 * cin].float()
    if layer.k_order == 1:      # k = (c // 64) * 9 * 64 + tap * 64 + c % 64
        w = w.reshape(n, cin // 64, 9, 64).permute(0, 2, 1, 3)
    return w.reshape(n, 3, 3, cin).permute(0, 3, 1, 2)


def shuffle(g, cout):
    """[B, 4*Cout, h, w] (phase p = 2*py + px in channels [p*Cout, (p+1)*Cout)) -> [B, Cout, 2h, 2w]."""
    B, _, h, w = g.shape
    return g.view(B, 2, 2, cout, h, w).permute(0, 3, 4, 1, 5, 2).reshape(B, cout, 2 * h, 2 * w)


@pytest.mark.parametrize("cin", [64, 512])
@pytest.mark.parametrize("hw", [(1, 1), (1, 9), (5, 7), (17, 22)])
@pytest.mark.parametrize("tc", [False, True], ids=["k_order0", "chunk_major"])
def test_polyphase_packing_is_the_transposed_conv(cin, hw, tc):
    torch.manual_seed(cin + hw[0] * 31 + hw[1])
    holder = _TransposedConvLayer(cin, cin // 2)
    layer = _transposed_layer(holder, torch.float32, tc)
    assert (layer.n, layer.ksize, layer.stride, layer.pad, layer.k_order) == (2 * cin, 3, 1, 1, int(tc))
    assert torch.equal(layer.bias, holder.transposed_conv2d.bias.detach().repeat(4))
    x = torch.randn(2, cin, *hw)
    with torch.no_grad():
        ref = F.relu(holder.transposed_conv2d(x))
        got = shuffle(F.relu(F.conv2d(x, unpack(layer, cin), layer.bias, padding=1)), cin // 2)
    assert got.shape == ref.shape == (2, cin // 2, 2 * hw[0], 2 * hw[1])
    err = float((got - ref).abs().max())
    print("cin", cin, "map", hw, "max-abs", err)
    assert err <= 1e-5


def test_polyphase_packing_uses_every_tap_once():
    """The 25 taps of every (ci, co) land in exactly one (phase, 3x3 position) and the other 11 positions are zero."""
    holder = _TransposedConvLayer(64, 32)
    with torch.no_grad():
        holder.transposed_conv2d.weight.copy_(torch.arange(1, 26, dtype=torch.float32).view(1, 1, 5, 5).expand(64, 32, 5, 5))
    w3 = unpack(_transposed_layer(holder, torch.float32, False), 64).view(4, 32, 64, 9)
    vals = w3[:, 0, 0, :].reshape(-1)
    assert sorted(int(v) for v in vals if v != 0) == list(range(1, 26))
    assert int((vals == 0).sum()) == 36 - 25


def _keys(m):
    return {k: tuple(v.shape) for k, v in m.state_dict().items()}


@pytest.mark.parametrize("over", [{}, {"recurrent_block_type": "convgru"}, {"num_encoders": 3}])
def test_construction_keys_and_strict_load(over):
    cfg = dict({"num_bins": 5, "use_upsample_conv": False}, **over)
    m = E2VIDRecurrent(cfg)
    up = E2VIDRecurrent(dict(cfg, use_upsample_conv=True))
    ne, bc = m.num_encoders, m.base_num_channels
    dec = {}
    for i in range(ne):
        cin = bc * 2 ** (ne - i)
        dec["unetrecurrent.decoders.%d.transposed_conv2d.weight" % i] = (cin, cin // 2, 5, 5)
        dec["unetrecurrent.decoders.%d.transposed_conv2d.bias" % i] = (cin // 2,)
    # every key outside the decoders is the upsample-conv model's; the decoders carry the reference's transposed keys
    other = {k: v for k, v in _keys(up).items() if ".decoders." not in k}
    assert _keys(m) == dict(other, **dec)
    sd = synth.random_state_dict_like(m.state_dict(), 5)
    m.load_state_dict(sd, strict=True)
    with pytest.raises(RuntimeError):
        up.load_state_dict(sd, strict=True)


def test_norm_bn_still_unsupported():
    with pytest.raises(NotImplementedError):
        E2VIDRecurrent({"num_bins": 5, "use_upsample_conv": False, "norm": "BN"})


def test_reference_transposed_decoder_is_the_module():
    torch.manual_seed(2)
    mod = nn.ConvTranspose2d(128, 64, 5, 2, 2, output_padding=1)
    sd = {"d.transposed_conv2d." + k: v.detach() for k, v in mod.state_dict().items()}
    x = torch.randn(2, 128, 5, 7)
    with torch.no_grad():
        ref = F.relu(mod(x))
    got = transposed_conv(sd, "d", x, "relu")
    assert got.shape == (2, 64, 10, 14)
    assert torch.equal(got, ref)


@pytest.mark.parametrize("over", [{}, {"recurrent_block_type": "convgru", "num_encoders": 3}])
def test_reference_step_is_the_oracle_schedule(over, monkeypatch):
    """e2vid_transposed_forward is the oracle's E2VIDRecurrent step with only the decoder layer exchanged: bit-equal to
    O.e2vid_recurrent_forward run with its upsample-conv decoder replaced by the transposed one."""
    from oracle import oracle_torch as O
    m = E2VIDRecurrent(dict({"num_bins": 5, "use_upsample_conv": False}, **over))
    sd = synth.random_state_dict_like(m.state_dict(), 8)
    ne = m.num_encoders
    g = torch.Generator().manual_seed(9)
    xs = [torch.randn(1, 5, 32, 48, generator=g) for _ in range(2)]
    with torch.no_grad():
        st, got = None, []
        for x in xs:
            img, st = e2vid_transposed_forward(sd, x, st, num_encoders=ne)
            got.append(img)
        monkeypatch.setattr(O, "upsample_conv", transposed_conv)
        st = None
        for x, a in zip(xs, got):
            img, st = O.e2vid_recurrent_forward(sd, x, st, num_encoders=ne)
            assert torch.equal(a, img)


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference tree not present")
@pytest.mark.parametrize("over", [{}, {"recurrent_block_type": "convgru", "num_encoders": 3}])
def test_transposed_decoders_vs_reference_live(over):
    """Our container's state_dict strictly loads into the reference's E2VIDRecurrent(use_upsample_conv=False), and the
    reference's UNetRecurrent frames (states carried) equal e2vid_transposed_forward's."""
    cfg = dict({"num_bins": 5, "use_upsample_conv": False}, **over)
    ours = E2VIDRecurrent(cfg)
    sd = synth.random_state_dict_like(ours.state_dict(), 11)
    R = ref_shim.reference_modules()
    ref = R.E2VIDRecurrent(dict(cfg)).eval()
    ref.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(12)
    st_ref = st_or = None
    ne = ours.num_encoders
    with ref_shim.cpu_mode(), torch.no_grad():
        for _ in range(3):
            x = torch.randn(1, 5, 48, 64, generator=g)
            a, st_ref = ref.unetrecurrent(x, st_ref)
            b, st_or = e2vid_transposed_forward(sd, x, st_or, num_encoders=ne)
            assert float((a - b).abs().max()) <= 1e-6
