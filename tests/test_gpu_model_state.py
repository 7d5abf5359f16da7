"""GPU: the state BlipITM derives from its parameters (weight operands, K/V buffers, captured CUDA graphs) follows every
parameter change, and a failed graph capture falls back to the eager pass."""
import copy
import warnings

import pytest
import torch

import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _tiny_model(tok, seed=11):
    from pnp_ovss_b200.blip_itm import BlipITM
    torch.manual_seed(seed)
    m = BlipITM(img_size=96, tokenizer=tok, vocab=30524, hidden=128, layers=3, heads=2, inter=256, vit_dim=64, vit_depth=2,
                vit_heads=2, max_pos=64).eval()
    with torch.no_grad():  # random init at std 0.02 gives near-uniform attention; widen it so the maps have structure
        for p in m.parameters():
            p.mul_(2.0)
    return m


def _case(dev, mode, seed=11):
    """(model on the GPU in GEMM mode `mode`, gradcam(*args) arguments)."""
    tok = synth.SyntheticWordPieceTokenizer()
    caps = ["A picture of cat aeroplane", "A picture of dog"]
    tokens = tok(caps, padding="max_length", max_length=500).to(dev)
    imgs = torch.randn(2, 3, 96, 96, generator=torch.Generator().manual_seed(3)).to(dev)
    m = _tiny_model(tok, seed).to(dev).requires_grad_(False)
    m.gemm_precision = mode
    return m, (imgs, caps, tokens, 1, 1)


@pytest.mark.parametrize("mode,bias", [("3xfp16", lambda m: m.visual_encoder.blocks[0].qkv.bias),
                                       ("3xtf32", lambda m: m.layer[0].crossattention.self.value.bias)],
                         ids=["3xfp16-vit-qkv-bias", "3xtf32-cross-value-bias"])
def test_inplace_bias_edit_after_a_graphed_pass_is_used(dev, mode, bias):
    """Both biases are copied into the cached operands (3xFP16 folds the ViT qkv bias into its operand columns; both modes
    keep one concatenated cross-attention K/V bias): an in-place edit must rebuild them, and the graphs that read them."""
    from pnp_ovss_b200 import ops
    m, args = _case(dev, mode)
    before, _ = m.gradcam(*args)                 # captures the encoder and text-pass graphs
    m.fp16_overflow_flag(dev).fill_(1)           # an overflow recorded before the weight change ...
    with torch.no_grad():
        bias(m).add_(0.5)
    got, out = m.gradcam(*args)
    fresh = copy.deepcopy(m)
    want, want_out = fresh.gradcam(*args)
    assert not torch.equal(got, before)
    assert torch.equal(got, want) and torch.equal(out, want_out)
    with pytest.raises(ops.PnpError):
        m.check_fp16_overflow()                  # ... is still reported
    fresh.check_fp16_overflow()                  # and a copy starts with a clear flag


def test_checkpoint_load_after_a_graphed_pass_is_used(dev):
    from pnp_ovss_b200.lavis_compat import export_lavis_state_dict
    m, args = _case(dev, "3xfp16")
    m.gradcam(*args)
    m.fp16_overflow_flag(dev).fill_(1)
    other, _ = _case(dev, "3xfp16", seed=12)
    m.load_lavis_checkpoint(export_lavis_state_dict(other))
    m.check_fp16_overflow()                      # a checkpoint load starts with a clear flag
    got, out = m.gradcam(*args)
    want, want_out = other.gradcam(*args)
    assert torch.equal(got, want) and torch.equal(out, want_out)


def test_failed_graph_capture_runs_the_pass_eagerly(dev, monkeypatch):
    m, args = _case(dev, "3xfp16")
    eager = copy.deepcopy(m)
    eager.USE_VIT_GRAPH = eager.USE_TEXT_GRAPH = False
    want, want_out = eager.gradcam(*args)

    def no_graph():
        raise RuntimeError("no graph capture here")

    monkeypatch.setattr(torch.cuda, "CUDAGraph", no_graph)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        results = [m.gradcam(*args) for _ in range(2)]
    msgs = sorted(str(w.message) for w in rec if issubclass(w.category, UserWarning))
    assert len(msgs) == 2, msgs                  # one per graph, not one per call
    assert msgs[0].startswith("encoder CUDA graph capture failed") and msgs[1].startswith("text-pass CUDA graph capture failed")
    for got, out in results:
        assert torch.equal(got, want) and torch.equal(out, want_out)
