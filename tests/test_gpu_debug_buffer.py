"""GPU: cfb_debug_buffer describes only the forwards whose workspace it can describe.  A bf16 batch of B >= 8 runs as two
half-batches, each with a workspace plan of its own (engine.cu, cfb_forward), so there the call is refused.  Below that,
and on the fp32 validation path at any B, every named intermediate lies inside cfb_workspace_bytes(B, T) and has the
size of its layout (test_gpu_subsampling.py checks the contents)."""
import ctypes

import pytest

import conformer_nemo_b200 as cn
from conformer_nemo_b200 import _lib
from oracle import conformer_oracle as oc

pytestmark = pytest.mark.gpu

CFG = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=176, n_heads=4)
T = 203


def conv_out(n):
    return (n - 1) // 2 + 1


def layout_bytes(B, esz):
    """Bytes of every named intermediate of a dense (B, T) forward; esz = bytes per activation element."""
    d, C, L, Dp = CFG.d_model, CFG.conv_channels, CFG.n_layers, CFG.n_heads * 64
    T1, F1 = conv_out(T), conv_out(CFG.feat_in)
    T2, F2 = conv_out(T1), conv_out(F1)
    Th, Fh = (T1 + 1) // 2, (F1 + 1) // 2
    N, P = B * T2, 2 * T2 - 1
    return {"y1": B * 4 * Th * Fh * C * esz, "y2": N * F2 * C * esz, "x": N * d * 4, "a": N * d * esz,
            "h": N * d * CFG.ff_expansion_factor * esz, "qkv": N * 4 * Dp * esz, "ctx": N * Dp * esz, "g": N * d * esz,
            "c": N * d * esz, "pe": P * d * esz, "pos": P * L * Dp * esz}


def run(precision, B):
    enc = cn.ConformerEncoder(feat_in=CFG.feat_in, n_layers=CFG.n_layers, d_model=CFG.d_model, n_heads=CFG.n_heads,
                              precision=precision)
    enc.load_state_dict(oc.random_state_dict(CFG, 3), strict=False)
    enc = enc.cuda().eval()
    enc.packed = False
    x, length = oc.synthetic_batch(B, CFG.feat_in, T, [T - 11 * b for b in range(B)], seed=4)
    enc(audio_signal=x.cuda(), length=length.cuda())
    return enc


@pytest.mark.parametrize("precision,B", [("bf16", 7), ("fp32_validate", 8)])
def test_debug_buffer_regions_lie_inside_the_workspace(precision, B):
    enc = run(precision, B)
    lib = _lib.load_library()
    ws = ctypes.c_size_t()
    _lib.check(lib.cfb_workspace_bytes(enc._handle, B, T, ctypes.byref(ws)), enc._handle, "cfb_workspace_bytes")
    for name, nbytes in layout_bytes(B, 4 if precision == "fp32_validate" else 2).items():
        off, got = ctypes.c_size_t(), ctypes.c_size_t()
        _lib.check(lib.cfb_debug_buffer(enc._handle, B, T, name.encode(), ctypes.byref(off), ctypes.byref(got)),
                   enc._handle, "cfb_debug_buffer")
        assert got.value == nbytes, (name, got.value, nbytes)
        assert off.value % 256 == 0 and off.value + got.value <= ws.value, (name, off.value, got.value, ws.value)
        assert enc.debug_buffer(B, T, name).numel() == nbytes, name


def test_debug_buffer_refuses_a_batch_that_runs_as_two_half_batches():
    enc = run("bf16", 8)
    with pytest.raises(ValueError, match="two half-batches"):
        enc.debug_buffer(8, T, "x")
