"""The synthesis hot path as one callable: decoder outputs -> audio -> multi-scale loss -> gradients.

This is decoder.py:106-125 + train.py:92-103,129 without the control network: the stage the
north star accelerates.  ``SynthStep`` owns static device buffers so that the whole forward +
backward can be captured once in a CUDA graph and replayed (SURVEY 7: configs 1 and 3 are launch
bound; one graph launch replaces ~30 kernel launches and all autograd bookkeeping).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import core
from . import functions as F_
from .shapes import SynthShapes, synthetic_inputs  # noqa: F401  (re-exported)


INPUT_NAMES = ("amp_raw", "dist_raw", "mag_raw", "pitch", "noise", "target")


class SynthStep:
    """Static-buffer runner of the hot path.  ``inputs`` are the decoder's raw outputs
    (harmonic_proj / noise_proj rows), pitch, the uniform noise draw and the target audio."""

    def __init__(self, shapes: SynthShapes, device="cuda", reverb_state: Optional[Dict[str, torch.Tensor]] = None):
        s = self.shapes = shapes
        dev = torch.device(device)
        f32 = dict(device=dev, dtype=torch.float32)
        # one contiguous block holds every input (each at a 16-byte-aligned offset), so that a host batch laid out the
        # same way (``pack_host``) reaches the device with ONE copy
        self._layout = [("amp_raw", (s.batch, s.frames, 1)), ("dist_raw", (s.batch, s.frames, s.n_harmonic)),
                        ("mag_raw", (s.batch, s.frames, s.n_bands)), ("pitch", (s.batch, s.frames, 1)),
                        ("noise", (s.batch, s.frames, s.block_size)), ("target", (s.batch, s.samples))]
        self.inputs, self._flat_in = self._alloc_inputs(dev)
        self.inputs["pitch"].fill_(220.0)
        self.reverb = None
        if s.reverb_length is not None:
            from .models.modules import Reverb
            self.reverb = Reverb(s.reverb_length, s.sample_rate).to(dev)
            if reverb_state is not None:
                self.reverb.load_state_dict(reverb_state)
        self._side_stream = torch.cuda.Stream(device=dev)
        self.loss = torch.zeros((), **f32)
        self.signal = None
        self.grads = None
        self._graph = None
        self._graph_fwd = None
        self._dist = None                  # set by enable_grad_allreduce (data-parallel training config)
        # the two synthesisers as one SynthPair node (noise CTAs per SM, 0 = the library's choice) where it applies,
        # else on two streams (None)
        self._pair_ctas = 0 if (core.harmonic_raw_supported(s.n_harmonic, s.block_size) and
                                F_.synth_pair_supported(s)) else None

    def _offsets(self):
        off, out = 0, []
        for name, shape in self._layout:
            n = 1
            for d in shape:
                n *= d
            out.append((name, shape, off, n))
            off += (n + 3) & ~3
        return out, off

    def _alloc_inputs(self, dev):
        offs, total = self._offsets()
        flat = torch.zeros(total, device=dev, dtype=torch.float32)
        return {name: flat[o:o + n].view(shape) for name, shape, o, n in offs}, flat

    def pack_host(self, host: Dict[str, torch.Tensor]) -> torch.Tensor:
        """A pinned host block with the batch in the device layout (what a data loader's collate function would fill)."""
        offs, total = self._offsets()
        flat = torch.zeros(total, dtype=torch.float32).pin_memory()
        for name, shape, o, n in offs:
            flat[o:o + n].view(shape).copy_(host[name])
        return flat

    # ---- data parallel: the shared parameters' gradients are averaged over the ranks (SURVEY 8e) -------
    def enable_grad_allreduce(self, dist, group=None, in_step: bool = True):
        """Voices are sharded over the ranks; the only shared parameters on this path are the reverb's
        (noise, decay, wet).  Their gradients are packed into one flat buffer and averaged with ONE NCCL all-reduce
        (op AVG) per step.

        ``in_step=True`` (default): the collective is part of run() and therefore a node of the captured CUDA graph.
        The backward is cut in two: the reverb PARAMETERS' backward first (the long convolution's kernel gradient, then
        the impulse's backward), then the all-reduce is queued on a communication stream while the convolution's signal
        gradient and the harmonic / noise / controls backward run on the compute streams; the step joins both at its
        end.  Every rank must then call run() / replay() the same number
        of times (a rank that steps alone waits for its peers forever): use ``local_only()`` around single-rank calls.
        ``in_step=False``: run() only packs; the caller queues ``allreduce_grads()`` after each step."""
        assert self.reverb is not None
        self._dist, self._group, self._in_step = dist, group, bool(in_step)
        self._sizes = [p.numel() for p in self.reverb.parameters()]
        self._flat = torch.zeros(sum(self._sizes), device=self.loss.device, dtype=torch.float32)
        self._comm_stream = torch.cuda.Stream(device=self.loss.device)

    def local_only(self):
        """Context manager: run()/forward_backward() without the collective (parity checks on one rank)."""
        step = self

        class _Local:
            def __enter__(self):
                self.saved = step._dist
                step._dist = None

            def __exit__(self, *a):
                step._dist = self.saved
        return _Local()

    def _pack(self, rev_grads):
        torch.cat([g.reshape(-1) for g in rev_grads], out=self._flat)
        return tuple(c.view(g.shape) for c, g in zip(self._flat.split(self._sizes), rev_grads))

    def allreduce_grads(self):
        """The collective of the ``in_step=False`` mode (a no-op otherwise: run() already contains it)."""
        if self._dist is not None and not self._in_step:
            self._dist.all_reduce(self._flat, op=self._dist.ReduceOp.AVG, group=self._group)

    # ---- the path -------------------------------------------------------------------------
    def _leaves(self):
        """Fresh leaf aliases of the differentiable buffers.  New leaves every call keep autograd's
        per-leaf bookkeeping on the stream of the current call, which CUDA-graph capture requires."""
        leaves = [self.inputs[k].detach().requires_grad_(True) for k in ("amp_raw", "dist_raw", "mag_raw")]
        if self.reverb is not None:
            leaves += [p.detach().requires_grad_(True) for p in
                       (self.reverb.noise, self.reverb.decay, self.reverb.wet)]
        return leaves

    def forward(self, leaves=None):
        """decoder.py:110-125: controls -> harmonic + filtered noise (+ reverb).  (B,N,1)"""
        i, s = self.inputs, self.shapes
        if leaves is None:
            leaves = [i["amp_raw"], i["dist_raw"], i["mag_raw"]]
            if self.reverb is not None:
                leaves += [self.reverb.noise, self.reverb.decay, self.reverb.wet]
        # The noise branch and the harmonic branch are independent until the mix (decoder.py:121).  Where the pair
        # applies, both synthesisers are one SynthPair node on the current stream: the noise kernel's persistent CTAs
        # and the oscillator bank share every SM in each direction.  Elsewhere the noise branch runs on a side stream
        # (autograd replays each node's backward on its forward stream, so the two backward branches overlap as well;
        # under capture both become parallel graph branches).
        cur = torch.cuda.current_stream()
        side = self._side_stream
        kernel = hspec = None
        noise = None
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            if self.reverb is not None:
                # the reverb's impulse depends on the reverb parameters only: it is built, and its spectrum computed,
                # on the side stream.  Autograd replays a node's backward on its forward stream, so the impulse's
                # backward (two small launches at the very end of the step) also lands beside the synthesisers'
                # backward instead of after it
                impulse = F_.ReverbImpulse.apply(leaves[3], leaves[4], leaves[5], self.reverb.t)
                taps = min(s.samples, s.reverb_length)
                kernel = impulse.reshape(1, s.reverb_length)[:, :taps]
                hspec = F_._ops.fftconv_spectrum(kernel.detach(), s.samples)
            if self._pair_ctas is None:
                # FilteredNoise.get_controls + forward in one launch
                noise = F_.FilteredNoiseFused.apply(leaves[2], i["noise"], None, -5.0)
        if self._pair_ctas is not None:
            harmonic, noise = F_.SynthPair.apply(leaves[0], leaves[1], leaves[2], i["pitch"], i["noise"], s.block_size,
                                                 s.sample_rate, -5.0, self._pair_ctas)
        elif core.harmonic_raw_supported(s.n_harmonic, s.block_size):
            # HarmonicSynth.get_controls + forward in one launch (the controls are the oscillator bank's prologue)
            harmonic = core.harmonic_synth_from_raw(leaves[0], leaves[1], i["pitch"], s.block_size, s.sample_rate)[0]
        else:
            _, _, weights = F_.HarmonicControlsWeights.apply(leaves[0], leaves[1], i["pitch"], float(s.sample_rate))
            harmonic, _ = core.harmonic_synth_frames(i["pitch"], weights, s.block_size, s.sample_rate)
        cur.wait_stream(side)
        noise.record_stream(cur)
        if self.reverb is not None:
            hspec.record_stream(cur)
            kernel.record_stream(cur)
            # decoder.py:121's `harmonic + noise` is formed by the reverb's first pass while it loads its input
            signal = F_.FFTConvolve.apply(harmonic.squeeze(-1), kernel, hspec, noise.squeeze(-1)).unsqueeze(-1)
        else:
            signal = harmonic + noise
        return signal

    def forward_backward(self):
        """train.py:89-103,129 on the synth part: loss and gradients of every leaf
        (amp_raw, dist_raw, mag_raw, reverb.noise, reverb.decay, reverb.wet)."""
        s = self.shapes
        leaves = self._leaves()
        signal = self.forward(leaves)
        # train.py:129 is loss.backward(): the loss node's upstream gradient is exactly 1, so the gradient w.r.t. the
        # reconstruction that the fused loss launch already produced goes straight into the synth chain's backward
        # (core.multiscale_spectral_loss would multiply it by that 1 in a separate elementwise launch)
        scales = [int(x) for x in s.scales]
        windows = F_.hann_windows_like_reference(scales, signal.device)
        loss, d_rec = F_._ops.mss_loss_fwd(self.inputs["target"], signal.detach().squeeze(-1), scales, float(s.overlap),
                                           windows, True)
        if self._dist is None or self.reverb is None:
            grads = torch.autograd.grad(signal, leaves, grad_outputs=d_rec.view_as(signal))
            return signal, loss, grads
        # data parallel: the reverb PARAMETERS' backward first (long convolution's kernel gradient -> impulse backward),
        # so that the collective on them is in flight while the convolution's signal gradient and the two
        # synthesisers' backward run.  Two autograd calls over the same gradient; the transform of d_rec is shared.
        g = d_rec.view_as(signal)
        with F_.fftconv_backward_part("kernel"):
            rev = self._pack(torch.autograd.grad(signal, leaves[3:], grad_outputs=g, retain_graph=True))
        cur = torch.cuda.current_stream()
        if self._in_step:
            comm = self._comm_stream
            comm.wait_stream(cur)
            with torch.cuda.stream(comm):
                self._dist.all_reduce(self._flat, op=self._dist.ReduceOp.AVG, group=self._group)
        with F_.fftconv_backward_part("signal"):
            front = torch.autograd.grad(signal, leaves[:3], grad_outputs=g)
        if self._in_step:
            cur.wait_stream(comm)
        return signal, loss, tuple(front) + rev

    # ---- eager / graph execution ---------------------------------------------------------
    def run(self):
        self.signal, loss, self.grads = self.forward_backward()
        self.loss = loss
        return loss

    def run_forward(self):
        with torch.no_grad():
            self.signal = self.forward()
        return self.signal

    def capture(self, forward_only: bool = False, warmup: int = 3):
        """Capture the step in a CUDA graph (after a few eager runs on a side stream so that lazily
        built tables and the allocator's pools exist before capture)."""
        fn = self.run_forward if forward_only else self.run
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            fn()
        if forward_only:
            self._graph_fwd = graph
        else:
            self._graph = graph
        return graph

    def release_graphs(self):
        """Drop every captured graph.  A graph that holds an NCCL node must be gone before its communicator is
        destroyed (destroy_process_group() waits for it otherwise)."""
        self._graph = self._graph_fwd = None
        self._pair = None
        import gc
        gc.collect()
        torch.cuda.synchronize()

    def replay(self, forward_only: bool = False):
        (self._graph_fwd if forward_only else self._graph).replay()

    # ---- host-fed execution: H2D of the next batch overlaps the current step -------------------
    def _staging(self):
        if getattr(self, "_stage", None) is None:
            self._stage = [{k: torch.empty_like(v) for k, v in self.inputs.items()} for _ in range(2)]
            self._copy_stream = torch.cuda.Stream()
            self._ready = [torch.cuda.Event(), torch.cuda.Event()]
            self._consumed = [torch.cuda.Event(), torch.cuda.Event()]
            self._slot = 0
            self._primed = False
        return self._stage

    def prefetch(self, host: Dict[str, torch.Tensor]) -> int:
        """Start the host->device copy of a batch (pinned tensors) on the copy stream into the idle
        staging set; returns the bytes queued.  The copy runs while the current step computes."""
        stage = self._staging()
        slot = self._slot
        n = 0
        self._copy_stream.wait_event(self._consumed[slot])       # staging set free again
        with torch.cuda.stream(self._copy_stream), torch.no_grad():
            for k in INPUT_NAMES:
                if k in host:
                    stage[slot][k].copy_(host[k], non_blocking=True)
                    n += host[k].numel() * host[k].element_size()
            self._ready[slot].record(self._copy_stream)
        self._primed = True
        return n

    def step_prefetched(self, forward_only: bool = False):
        """Run one step on the batch most recently handed to ``prefetch``: wait for its copy, move it
        into the graph's static inputs (device-to-device), replay."""
        assert getattr(self, "_primed", False), "call prefetch() first"
        slot = self._slot
        cur = torch.cuda.current_stream()
        cur.wait_event(self._ready[slot])
        with torch.no_grad():
            for k, v in self._stage[slot].items():
                self.inputs[k].copy_(v, non_blocking=True)
        self._consumed[slot].record(cur)
        self._slot ^= 1
        graph = self._graph_fwd if forward_only else self._graph
        if graph is not None:
            graph.replay()
        elif forward_only:
            self.run_forward()
        else:
            self.run()

    # ---- host-fed execution without device-side copies: several input sets, one captured graph each -------
    def capture_pair(self, warmup: int = 3, sets: int = 2):
        """Capture the forward+backward step once per set of static input buffers (``sets`` of them, two by default).
        ``feed`` copies a host batch straight into the next idle set on the copy stream while the other sets' graphs
        run; ``step_fed`` replays the graph of the oldest fed set.  No staging buffers and no device-to-device copy: per
        step the GPU sees one H2D transfer (copy engine) and one graph launch.  With n sets the copy of a batch has n - 1
        step times to arrive and the host may queue n - 1 steps ahead, which absorbs jitter of the host and of the
        link; two sets already overlap copy and compute when neither stalls."""
        assert sets >= 2
        first, first_flat = self.inputs, self._flat_in
        entries = [(first, first_flat)]
        for _ in range(sets - 1):
            inputs, flat = self._alloc_inputs(first_flat.device)
            flat.copy_(first_flat)
            entries.append((inputs, flat))
        self._pair = []
        for inputs, flat in entries:
            self.inputs = inputs
            graph = self.capture(forward_only=False, warmup=warmup)
            self._pair.append({"inputs": inputs, "flat": flat, "graph": graph, "signal": self.signal, "loss": self.loss,
                               "grads": self.grads})
        self.inputs = first
        self._graph = self._pair[0]["graph"]
        self._copy_stream2 = torch.cuda.Stream()
        self._fed = [torch.cuda.Event() for _ in range(sets)]
        self._used = [torch.cuda.Event() for _ in range(sets)]
        self._fill = 0                     # next set to feed
        self._next = 0                     # next set to run
        self._loss_host = torch.zeros(sets, dtype=torch.float32).pin_memory()
        self._loss_ready = [torch.cuda.Event() for _ in range(sets)]
        self._loss_done = [torch.cuda.Event() for _ in range(sets)]
        self._loss_stream = torch.cuda.Stream()
        return self._pair

    def feed(self, host) -> int:
        """Host batch -> the next idle input set, on the copy stream; returns the bytes queued.  ``host`` is a dict of
        pinned tensors (one copy each) or one pinned block from ``pack_host`` (a single copy).  At most
        ``sets - 1`` batches may be fed ahead of the step that is running."""
        k = self._fill
        self._copy_stream2.wait_event(self._used[k])             # the graph that last read this set has finished
        n = 0
        with torch.cuda.stream(self._copy_stream2), torch.no_grad():
            if isinstance(host, torch.Tensor):
                self._pair[k]["flat"].copy_(host, non_blocking=True)
                n = host.numel() * host.element_size()
            else:
                for name in INPUT_NAMES:
                    if name in host:
                        self._pair[k]["inputs"][name].copy_(host[name], non_blocking=True)
                        n += host[name].numel() * host[name].element_size()
            self._fed[k].record(self._copy_stream2)
        self._fill = (k + 1) % len(self._pair)
        return n

    def step_fed(self) -> int:
        """Run the step on the oldest fed set; returns its index (for ``loss_to_host`` / ``read_loss``)."""
        k = self._next
        cur = torch.cuda.current_stream()
        cur.wait_event(self._fed[k])
        e = self._pair[k]
        e["graph"].replay()
        self._used[k].record(cur)
        self.inputs, self.signal, self.loss, self.grads = e["inputs"], e["signal"], e["loss"], e["grads"]
        self._next = (k + 1) % len(self._pair)
        return k

    def loss_to_host(self, k: int):
        """Queue the device->host read of set k's loss (after the step, and after the gradient all-reduce if any).
        The 4-byte copy goes on its own stream, so that it never sits between two graph launches on the compute stream
        (where a driver that serves both copy directions with one engine would make it, and the next step, wait for the
        host->device transfer of a later batch; measured: no difference on the boxes of this round)."""
        cur = torch.cuda.current_stream()
        self._loss_done[k].record(cur)
        self._loss_stream.wait_event(self._loss_done[k])
        with torch.cuda.stream(self._loss_stream), torch.no_grad():
            self._loss_host[k:k + 1].copy_(self._pair[k]["loss"].detach().reshape(1), non_blocking=True)
            self._loss_ready[k].record(self._loss_stream)

    def read_loss(self, k: int) -> float:
        self._loss_ready[k].synchronize()
        return float(self._loss_host[k])

    def load_inputs(self, host: Dict[str, torch.Tensor], non_blocking: bool = True) -> int:
        """Copy a batch from (pinned) host tensors into the static buffers; returns bytes copied."""
        n = 0
        with torch.no_grad():
            for k in INPUT_NAMES:
                if k in host:
                    self.inputs[k].copy_(host[k], non_blocking=non_blocking)
                    n += host[k].numel() * host[k].element_size()
        return n
