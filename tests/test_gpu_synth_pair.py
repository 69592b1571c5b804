"""The synth pair (SynthPair: the oscillator bank launched beside the persistent filtered-noise kernel) computes the
same bits as the two Functions it replaces, eagerly and replayed from a CUDA graph, and SynthStep with it matches
SynthStep on two streams."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BENCH = dict(frames=400, block_size=160, n_harmonic=100, n_bands=65, sample_rate=16000)


def _shapes(batch, reverb_length=None):
    from ddsp_pytorch_b200.shapes import SynthShapes
    return SynthShapes(batch=batch, reverb_length=reverb_length, **BENCH)


def test_pair_applies_to_the_benchmark_batches_only():
    from ddsp_pytorch_b200 import functions as F_
    assert F_.synth_pair_supported(_shapes(64)) and F_.synth_pair_supported(_shapes(16))
    assert F_.synth_pair_supported(_shapes(64), 1) and F_.synth_pair_supported(_shapes(64), 2)
    # too few frames to give every noise CTA a full sweep: the two-stream layout
    assert not F_.synth_pair_supported(_shapes(2))
    assert not F_.synth_pair_supported(_shapes(64), 3)


def _inputs(batch, seed):
    from ddsp_pytorch_b200.shapes import synthetic_inputs
    host = synthetic_inputs(_shapes(batch), seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    n = batch * BENCH["frames"] * BENCH["block_size"]
    dev = {k: v.cuda() for k, v in host.items()}
    dev["g_h"] = torch.randn(batch, n // batch, 1, generator=g).cuda()
    dev["g_n"] = torch.randn(batch, n // batch, 1, generator=g).cuda()
    return dev


def _separate(x):
    from ddsp_pytorch_b200 import core, functions as F_
    leaves = [x[k].detach().requires_grad_(True) for k in ("amp_raw", "dist_raw", "mag_raw")]
    h = core.harmonic_synth_from_raw(leaves[0], leaves[1], x["pitch"], BENCH["block_size"], BENCH["sample_rate"])[0]
    n = F_.FilteredNoiseFused.apply(leaves[2], x["noise"], None, -5.0)
    grads = torch.autograd.grad((h, n), leaves, grad_outputs=(x["g_h"], x["g_n"]))
    return [h.detach(), n.detach(), *grads]


def _pair(x, ctas):
    from ddsp_pytorch_b200 import functions as F_
    leaves = [x[k].detach().requires_grad_(True) for k in ("amp_raw", "dist_raw", "mag_raw")]
    h, n = F_.SynthPair.apply(leaves[0], leaves[1], leaves[2], x["pitch"], x["noise"], BENCH["block_size"],
                              BENCH["sample_rate"], -5.0, ctas)
    grads = torch.autograd.grad((h, n), leaves, grad_outputs=(x["g_h"], x["g_n"]))
    return [h.detach(), n.detach(), *grads]


NAMES = ("harmonic", "noise", "d_amp_raw", "d_dist_raw", "d_mag_raw")


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [64, 16, 7])
@pytest.mark.parametrize("ctas", [0, 1, 2])
def test_pair_matches_the_two_functions_bit_for_bit(batch, ctas):
    x = _inputs(batch, seed=batch)
    ref = _separate(x)
    got = _pair(x, ctas)
    torch.cuda.synchronize()
    for name, a, b in zip(NAMES, got, ref):
        assert torch.equal(a, b), f"{name} differs at batch {batch}, {ctas} CTAs per SM"


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [64, 16, 7])
def test_pair_replayed_from_a_graph_matches_the_two_functions(batch):
    x = _inputs(batch, seed=100 + batch)
    ref = _separate(x)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _pair(x, 0)                                   # warm-up: tables and allocator pools exist before capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _pair(x, 0)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    for name, a, b in zip(NAMES, out, ref):
        assert torch.equal(a, b), f"{name} differs after graph replay at batch {batch}"


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [64, 16])
def test_step_with_the_pair_matches_the_two_stream_step(batch):
    """The whole step, graph-replayed: audio, loss and all six gradients.  A missing edge from the noise kernel to the
    reverb's first pass (forward) or to the step's end (backward) shows up here as a difference."""
    from ddsp_pytorch_b200.hotpath import SynthStep
    from ddsp_pytorch_b200.shapes import synthetic_inputs
    shapes = _shapes(batch, reverb_length=16000)
    host = {k: v.pin_memory() for k, v in synthetic_inputs(shapes, seed=5).items()}
    outs = []
    for ctas in (None, 0):
        torch.manual_seed(0)
        step = SynthStep(shapes, "cuda")
        assert step._pair_ctas == 0
        step._pair_ctas = ctas
        step.load_inputs(host)
        step.capture(forward_only=False)
        step.replay()
        torch.cuda.synchronize()
        res = [step.signal.detach().clone(), step.loss.detach().clone()] + [g.detach().clone() for g in step.grads]
        step.capture(forward_only=True)
        step.replay(forward_only=True)
        torch.cuda.synchronize()
        res.append(step.signal.detach().clone())
        outs.append(res)
    for i, (a, b) in enumerate(zip(*outs)):
        assert torch.equal(a, b), f"output {i} differs between the pair and the two-stream step at batch {batch}"
