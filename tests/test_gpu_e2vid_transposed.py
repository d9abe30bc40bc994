"""GPU: E2VIDRecurrent with use_upsample_conv=False -- TransposedConvLayer decoders run as one 3x3 phase convolution on
the low-resolution map (bde_gemm) followed by bde_shuffle2x_sum, which also adds the next decoder's skip.

* bde_shuffle2x_sum against a torch restatement, bit-exact in fp32 and bf16, with and without skip;
* frames and states against the CPU fp32 restatement (tests/e2vid_transposed_ref.py) over several steps with states
  carried (ConvLSTM / 4 encoders, ConvGRU / 3);
* the kernels one step launches: one shuffle per decoder, no bilinear upsample, the TMA conv kernel for the decoder
  convolutions at the e2vid16 size."""
import pytest
import torch

from bde2vid_b200 import ops, synth
from e2vid_transposed_ref import e2vid_transposed_forward

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {"fp32": 2e-4, "bf16": 2e-3}


def ref_shuffle(g, skip, c):
    n, h, w, _ = g.shape
    out = g.view(n, h, w, 2, 2, c).permute(0, 1, 3, 2, 4, 5).reshape(n, 2 * h, 2 * w, c)
    return out if skip is None else out + skip


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("with_skip", [False, True], ids=["noskip", "skip"])
@pytest.mark.parametrize("shape", [(1, 1, 1, 32), (1, 1, 1, 512), (2, 3, 5, 32), (3, 4, 7, 64), (2, 17, 22, 256),
                                   (1, 6, 10, 512), (2, 9, 11, 8)])
def test_shuffle2x_sum_kernel(dtype, with_skip, shape):
    n, h, w, c = shape
    g = torch.randn(n, h, w, 4 * c, device=DEV).to(dtype)
    skip = torch.randn(n, 2 * h, 2 * w, c, device=DEV).to(dtype) if with_skip else None
    buf = torch.full((n + 1, 2 * h, 2 * w, c), float("nan"), device=DEV, dtype=dtype)    # [n] guards against overruns
    ops.shuffle2x_sum(g, skip, n, h, w, c, buf[:n])
    torch.cuda.synchronize()
    assert torch.equal(buf[:n], ref_shuffle(g, skip, c))
    assert torch.isnan(buf[n]).all()


def test_shuffle2x_sum_rejects_bad_channels():
    g = torch.zeros(1, 2, 2, 48, device=DEV)
    with pytest.raises(RuntimeError):
        ops.shuffle2x_sum(g, None, 1, 2, 2, 12, torch.zeros(1, 4, 4, 12, device=DEV))


CONFIGS = {"lstm_ne4": {"num_encoders": 4}, "gru_ne3": {"recurrent_block_type": "convgru", "num_encoders": 3}}


def _model(over, precision, seed):
    from bde2vid_b200.e2vid import E2VIDRecurrent
    model = E2VIDRecurrent(dict({"num_bins": 5, "use_upsample_conv": False}, **over))
    sd = synth.random_state_dict_like(model.state_dict(), seed)
    model.load_state_dict(sd, strict=True)
    model = model.eval().to(DEV)
    model.unetrecurrent.precision = precision
    return model, sd


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("size", [(2, 64, 96), (1, 48, 80)], ids=["B2_64x96", "B1_48x80"])
@pytest.mark.parametrize("cfg", list(CONFIGS), ids=list(CONFIGS))
def test_transposed_decoders_vs_reference_port(cfg, size, precision):
    """Four steps with states carried; after step 1 the states go back in the reference's layout (ConvLSTM (h, c)
    NCHW tuples, ConvGRU NCHW tensors)."""
    model, sd = _model(CONFIGS[cfg], precision, 21)
    ne, lstm = model.num_encoders, model.recurrent_block_type == "convlstm"
    B, H, W = size
    gen = torch.Generator().manual_seed(22)
    st, st_ref = None, None
    with torch.no_grad():
        for i in range(4):
            x = torch.randn(B, 5, H, W, generator=gen) * (torch.rand(B, 5, H, W, generator=gen) < 0.5)
            ref, st_ref = e2vid_transposed_forward(sd, x, st_ref, num_encoders=ne)
            if i == 2:
                st = [(s.h, s.c) if lstm else s.h for s in st]
            img, st = model.unetrecurrent(x.to(DEV), st)
            assert img.shape == (B, 1, H, W) and img.dtype == torch.float32
            err = float((img.cpu() - ref).abs().max())
            print(cfg, size, precision, "step", i, "max-abs", err)
            assert err <= TOL[precision]
            for a, b in zip(st, st_ref):
                got, want = (a.c, b[1]) if lstm else (a.h, b)
                assert got.shape == want.shape
                assert float((got.cpu() - want).abs().max()) <= (1e-4 if precision == "fp32" else 3e-2)


def _kernels_in_order(fn):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == DeviceType.CUDA]
    return [e.name for e in sorted(evs, key=lambda e: e.time_range.start)]


@pytest.mark.parametrize("size", [(2, 64, 96), (16, 272, 352)], ids=["B2_64x96", "B16_272x352"])
def test_transposed_decoder_route(size):
    """One step launches one shuffle per decoder and no bilinear upsample; each shuffle follows its decoder GEMM, which
    at the e2vid16 size (every decoder input at least 8 x 8) is the TMA-fed tcgen05 conv kernel."""
    model, _ = _model({}, "bf16", 23)
    ne = model.num_encoders
    B, H, W = size
    x = torch.randn(B, 5, H, W, device=DEV)
    with torch.no_grad():
        model({"events": x})
        names = _kernels_in_order(lambda: model({"events": x}))
    assert not any("upsample2x_sum" in n for n in names)
    at = [i for i, n in enumerate(names) if "shuffle2x_sum_kernel" in n]
    assert len(at) == ne, names
    if H >= 8 * 2 ** ne and W >= 8 * 2 ** ne:
        for i in at:
            assert "conv_tma_kernel" in names[i - 1], names[i - 1]
