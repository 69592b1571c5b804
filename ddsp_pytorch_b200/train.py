"""Data-parallel training harness for the decoder / autoencoder models (SURVEY 8f rank 4).

The reference's ``train.py`` is a single-device, module-level script around a Lightning data module
(``train.py:45-164``, ``ddsp/data.py:9-74``).  This module gives the same training recipe as a library +
``python -m ddsp_pytorch_b200.train`` entry point that runs one process per GPU under ``torchrun``:

* data: the reference's on-disk format (``signals.npy``, ``pitchs.npy``, ``loudness.npy``, ``mfccs.npy`` in one
  directory, ``data.py:13-16``), memory-mapped, batches with the reference's keys (``sig``, ``pitch``,
  ``loudness``, ``mfcc``; the last MFCC frame dropped as at ``data.py:25``); ``tools/extract_features.py`` writes a
  dataset's ``loudness.npy`` and ``mfccs.npy`` from its ``signals.npy`` on the GPU (``core.extract_features``), and
  with ``--pitch`` its ``pitchs.npy`` by YIN (``core.extract_pitch_yin``; the reference used CREPE, which is not part of
  this repo), so recordings alone make a dataset; ``write_synthetic_dataset`` makes a dataset of that format with
  synthetic features;
* every rank takes a disjoint, equal slice of each global batch (``distributed.shard_range``), batches are
  staged through pinned host memory one step ahead on a copy stream;
* step: loudness standardised with the training-set statistics (``train.py:86``), model forward, fused
  multi-scale spectral loss (``train.py:70-76,92-103`` in one kernel family), backward, ONE bucketed all-reduce
  (mean) of all parameter gradients over NCCL (``distributed.GradBucket``), Adam (``train.py:63``);
* ``state.pth`` (best running-mean loss, ``train.py:141-147``) and ``config.yaml`` next to it, written by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import threading
import queue
from pathlib import Path
from typing import Dict, Iterator, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist

from . import core
from .distributed import GradBucket, global_mean, shard_range

NPY_FILES = ("signals", "pitchs", "loudness", "mfccs")


class NpyDataset(torch.utils.data.Dataset):
    """``ddsp/data.py:9-33``: four ``.npy`` arrays in ``out_dir`` indexed by example; memory-mapped."""

    def __init__(self, out_dir):
        out_dir = Path(out_dir)
        self.signals, self.pitchs, self.loudness, self.mfccs = (
            np.load(out_dir / f"{name}.npy", mmap_mode="r") for name in NPY_FILES)
        n = self.signals.shape[0]
        if not (self.pitchs.shape[0] == self.loudness.shape[0] == self.mfccs.shape[0] == n):
            raise ValueError("the four .npy files do not hold the same number of examples")

    def __len__(self) -> int:
        return self.signals.shape[0]

    def __getitem__(self, idx) -> Dict[str, torch.Tensor]:
        return self.batch(np.asarray([idx]), squeeze=True)

    def batch(self, indices: np.ndarray, squeeze: bool = False) -> Dict[str, torch.Tensor]:
        """Examples ``indices`` stacked (``data.py:59-73``'s collate): sig (B,N), pitch / loudness (B,T,1),
        mfcc (B,T,n_mfcc) without the extractor's extra last frame."""
        order = np.sort(indices)                     # ascending reads from the memory map
        out = {
            "sig": torch.from_numpy(np.ascontiguousarray(self.signals[order], dtype=np.float32)),
            "pitch": torch.from_numpy(np.ascontiguousarray(self.pitchs[order], dtype=np.float32)).unsqueeze(-1),
            "loudness": torch.from_numpy(np.ascontiguousarray(self.loudness[order], dtype=np.float32)).unsqueeze(-1),
            "mfcc": torch.from_numpy(np.ascontiguousarray(self.mfccs[order][:, :-1, :], dtype=np.float32)),
        }
        return {k: v[0] for k, v in out.items()} if squeeze else out


def write_synthetic_dataset(out_dir, n_examples: int, sample_rate: int = 16000, block_size: int = 160,
                            seconds: float = 4.0, n_mfcc: int = 30, seed: int = 0) -> Path:
    """A dataset in the reference's format (``preprocess.py:77-88`` writes the same four arrays) made of
    harmonic tones with a slow vibrato and a loudness envelope, so that a model can actually fit it.  The pitch and
    loudness arrays are the synthesis controls; ``mfccs.npy`` is standard-normal noise.  Run
    ``tools/extract_features.py --overwrite`` on the directory to replace loudness and MFCCs by the features of the
    signals themselves."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(seed)
    frames = int(seconds * sample_rate) // block_size
    n = frames * block_size
    t = np.arange(n, dtype=np.float64) / sample_rate
    tf = t[::block_size]
    signals = np.empty((n_examples, n), np.float32)
    pitchs = np.empty((n_examples, frames), np.float32)
    loudness = np.empty((n_examples, frames), np.float32)
    mfccs = rng.standard_normal((n_examples, frames + 1, n_mfcc)).astype(np.float32)
    for i in range(n_examples):
        f0 = rng.uniform(110.0, 660.0)
        vib = 1.0 + 0.01 * np.sin(2 * np.pi * rng.uniform(3, 7) * t)
        env = 0.1 + 0.4 * (0.5 + 0.5 * np.sin(2 * np.pi * rng.uniform(0.2, 1.0) * t + rng.uniform(0, 6.28)))
        phase = 2 * np.pi * np.cumsum(f0 * vib) / sample_rate
        tone = sum(np.sin(k * phase) / k for k in range(1, 9) if k * f0 * 1.01 < sample_rate / 2)
        signals[i] = (env * tone / 2.0).astype(np.float32)
        pitchs[i] = (f0 * vib[::block_size]).astype(np.float32)
        loudness[i] = (20 * np.log10(env[::block_size]) - 10 + 0.0 * tf).astype(np.float32)
    for name, arr in zip(NPY_FILES, (signals, pitchs, loudness, mfccs)):
        np.save(out_dir / f"{name}.npy", arr)
    return out_dir


def loudness_stats(dataset: NpyDataset, batch: int) -> tuple:
    """``core.mean_std_loudness`` (``ddsp/core.py:14-24``) over consecutive batches of the training set."""
    n = len(dataset) // batch * batch
    batches = ({"loudness": torch.from_numpy(np.array(dataset.loudness[i:i + batch], dtype=np.float32))}
               for i in range(0, n, batch))
    return core.mean_std_loudness(batches)


class ShardedLoader:
    """Epoch iterator: a seeded global permutation (identical on all ranks), ``drop_last`` global batches
    (``data.py:45-49``), of which this rank reads its contiguous slice.  A worker thread reads and pins the next
    batches while the GPU works; ``__iter__`` yields device tensors whose H2D copy ran on ``copy_stream``."""

    def __init__(self, dataset: NpyDataset, global_batch: int, rank: int, world: int, device, seed: int = 0,
                 depth: int = 2):
        self.dataset, self.global_batch, self.device, self.seed, self.depth = dataset, global_batch, device, seed, depth
        self.lo, self.hi = shard_range(global_batch, world, rank)
        self.epoch = 0
        self.copy_stream = torch.cuda.Stream(device=device) if torch.device(device).type == "cuda" else None

    def __len__(self) -> int:
        return len(self.dataset) // self.global_batch

    def indices(self, epoch: int, step: int) -> np.ndarray:
        perm = np.random.default_rng(self.seed + epoch).permutation(len(self.dataset))
        return perm[step * self.global_batch + self.lo: step * self.global_batch + self.hi]

    def __iter__(self) -> Iterator[Dict[str, torch.Tensor]]:
        epoch, self.epoch = self.epoch, self.epoch + 1
        q: "queue.Queue" = queue.Queue(maxsize=self.depth)

        stop = threading.Event()

        def produce():
            for step in range(len(self)):
                if stop.is_set():
                    return
                host = self.dataset.batch(self.indices(epoch, step))
                if self.copy_stream is not None:
                    host = {k: v.pin_memory() for k, v in host.items()}
                while not stop.is_set():
                    try:
                        q.put(host, timeout=0.1)
                        break
                    except queue.Full:
                        continue
            if not stop.is_set():
                q.put(None)

        worker = threading.Thread(target=produce, daemon=True)
        worker.start()
        try:
            while True:
                host = q.get()
                if host is None:
                    return
                if self.copy_stream is None:
                    yield host
                    continue
                with torch.cuda.stream(self.copy_stream):
                    dev = {k: v.to(self.device, non_blocking=True) for k, v in host.items()}
                torch.cuda.current_stream(self.device).wait_stream(self.copy_stream)
                for v in dev.values():
                    v.record_stream(torch.cuda.current_stream(self.device))
                yield dev
        finally:                                     # the consumer left (break at the step limit): release the worker
            stop.set()
            while not q.empty():
                try:
                    q.get_nowait()
                except queue.Empty:
                    break
            worker.join(timeout=5)


class Trainer:
    """One rank of the data-parallel job.  ``model`` is a ``DDSPDecoder`` / ``DDSPAutoencoder`` on ``device``
    with identical initial parameters on every rank (same seed, or broadcast by ``sync_parameters``)."""

    def __init__(self, model: torch.nn.Module, scales: Sequence[int], overlap: float, lr: float,
                 mean_loudness: float, std_loudness: float, device, group=None, use_graph: bool = False,
                 graph_after: int = 3):
        self.model, self.scales, self.overlap = model, [int(s) for s in scales], float(overlap)
        self.mean_loudness, self.std_loudness = float(mean_loudness), float(std_loudness)
        self.device, self.group = device, group
        self.params = [p for p in model.parameters() if p.requires_grad]
        self.opt = torch.optim.Adam(self.params, lr=lr, fused=bool(self.params and self.params[0].is_cuda))
        self.bucket = GradBucket([p.shape for p in self.params], device, group=group)
        self.step_count = 0
        self.use_graph, self.graph_after, self.graph = use_graph, graph_after, None
        self.static_batch: Dict[str, torch.Tensor] = {}
        self.static_loss: Optional[torch.Tensor] = None

    def sync_parameters(self) -> None:
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            for t in list(self.model.parameters()) + list(self.model.buffers()):
                dist.broadcast(t.data, src=0, group=self.group)

    def loss_of(self, batch: Dict[str, torch.Tensor]) -> torch.Tensor:
        batch = dict(batch)
        batch["loudness"] = (batch["loudness"] - self.mean_loudness) / self.std_loudness       # train.py:86
        rec = self.model(batch)["signal"].squeeze(-1)
        return core.multiscale_spectral_loss(batch["sig"], rec, self.scales, self.overlap)

    def _all_reduce_grads(self) -> None:
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in self.params]
            for p, g in zip(self.params, self.bucket.all_reduce_mean(grads)):
                p.grad = g.clone() if p.grad is None else p.grad.copy_(g)

    def train_step(self, batch: Dict[str, torch.Tensor]) -> torch.Tensor:
        """Forward, backward, gradient all-reduce (mean over ranks = gradient of the global-batch mean loss),
        Adam.  Returns the global-batch loss (a device scalar, no host sync).

        With ``use_graph`` the forward + backward of the whole model (~350 launches, host-bound in eager mode)
        is captured once into a CUDA graph after ``graph_after`` eager steps and replayed on static input
        buffers; the all-reduce and the optimizer stay outside the graph."""
        self.step_count += 1
        if self.use_graph and self.graph is None and self.step_count > self.graph_after:
            self._capture(batch)
        if self.graph is not None and all(batch[k].shape == v.shape for k, v in self.static_batch.items()):
            for k, v in self.static_batch.items():
                v.copy_(batch[k], non_blocking=True)
            self.graph.replay()
            loss = self.static_loss
        else:
            loss = self.loss_of(batch)
            self.opt.zero_grad(set_to_none=self.graph is None)
            loss.backward()
        self._all_reduce_grads()
        self.opt.step()
        return global_mean(loss, self.group)

    def _capture(self, batch: Dict[str, torch.Tensor]) -> None:
        keys = [k for k in ("sig", "pitch", "loudness", "mfcc") if k in batch]
        self.static_batch = {k: batch[k].clone() for k in keys}
        self.opt.zero_grad(set_to_none=True)             # the graph owns the gradient buffers from here on
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):                    # one un-captured pass on the capture stream's allocator state
            self.loss_of(self.static_batch).backward()
        torch.cuda.current_stream(self.device).wait_stream(side)
        self.opt.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.static_loss = self.loss_of(self.static_batch)
            self.static_loss.backward()
        self.graph = graph

    @torch.no_grad()
    def evaluate(self, loader) -> float:
        total, count = torch.zeros((), device=self.device), 0
        for batch in loader:
            total += global_mean(self.loss_of(batch), self.group)
            count += 1
        return float(total / max(count, 1))


def build_model(name: str, kwargs: dict) -> torch.nn.Module:
    """``train.py:34-42``."""
    from .models.decoder import DDSPDecoder
    from .models.encoder import DDSPAutoencoder
    if name in ("decoder", "single-inst-decoder"):           # config.yaml:14 / this CLI's short name
        return DDSPDecoder(**kwargs)
    if name in ("autoencoder", "mfcc-autoencoder"):          # autoencoder.yaml:14
        return DDSPAutoencoder(**kwargs)
    raise ValueError(f"invalid model name: {name}")


def run(args) -> dict:
    """The job of one rank; returns a small report (rank 0's is printed by ``main``)."""
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    torch.manual_seed(args.seed)                                    # same initial parameters on every rank

    train_dir = Path(args.data) / "train" if (Path(args.data) / "train").is_dir() else Path(args.data)
    data = NpyDataset(train_dir)
    frames, n = data.pitchs.shape[1], data.signals.shape[1]
    kwargs = dict(hidden_size=args.hidden_size, n_harmonic=args.n_harmonic, n_bands=args.n_bands,
                  sample_rate=args.sample_rate, block_size=n // frames, has_reverb=not args.no_reverb)
    model = build_model(args.model, kwargs).to(device)
    # modules.py:119-123 draws the noise with the CPU generator and moves it (17 ms of host time per step at
    # batch 64, more than the GPU step); the default here is to draw on the device, --cpu-noise restores it
    model.noise_synth.device_noise = not args.cpu_noise
    if args.stock_control_net:                                      # A/B: cuBLAS / cuDNN layers as in the reference
        core.to_stock_layers(model)
    mean_l, std_l = loudness_stats(data, args.batch)
    trainer = Trainer(model, args.scales, args.overlap, args.lr, mean_l, std_l, device, use_graph=not (args.no_graph or args.cpu_noise))      # a CPU draw cannot be captured
    trainer.sync_parameters()
    # parameters are identical on every rank (same seed + broadcast); the noise draws must NOT be: with one seed all
    # ranks would excite voices i and i + B/world with the same noise, which a single-GPU run of the batch never does
    torch.manual_seed(args.seed + 1000 * (rank + 1))
    if device.type == "cuda":
        torch.cuda.manual_seed(args.seed + 1000 * (rank + 1))
    loader = ShardedLoader(data, args.batch, rank, world, device, seed=args.seed)
    if len(loader) == 0:
        raise ValueError(f"dataset of {len(data)} examples is smaller than the global batch {args.batch}")

    out_dir = Path(args.root) / args.name
    if rank == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
        ref_names = {"decoder": "single-inst-decoder", "autoencoder": "mfcc-autoencoder"}     # train.py:37-40, config.yaml:14
        config = {"model": {"name": ref_names[args.model], "kwargs": kwargs},
                  "data": {"mean_loudness": mean_l, "std_loudness": std_l},
                  "train": {"scales": list(args.scales), "overlap": args.overlap, "lr": args.lr, "batch": args.batch,
                            "steps": args.steps, "world_size": world}}
        try:
            import yaml
            (out_dir / "config.yaml").write_text(yaml.safe_dump(config))
        except ImportError:
            (out_dir / "config.json").write_text(json.dumps(config, indent=1))

    best, running, seen, first, last = float("inf"), 0.0, 0, None, None
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    timed_from = min(args.warmup, max(args.steps - 1, 0))
    done = 0
    while done < args.steps:
        for batch in loader:
            if done == timed_from:
                torch.cuda.synchronize()
                start.record()
            loss = trainer.train_step(batch)
            done += 1
            if done % args.log_every == 0 or done == args.steps:
                value = float(loss)                                  # the only host sync of the loop
                first = value if first is None else first
                last = value
                seen += 1
                running += (value - running) / seen                 # train.py:136-139
                if seen >= args.ckpt_window or done == args.steps:  # train.py:141-151: compare the window's mean,
                    if rank == 0 and running < best:                # keep the best, start a new window
                        best = running
                        torch.save(model.state_dict(), out_dir / "state.pth")
                    running, seen = 0.0, 0
            if done >= args.steps:
                break
    end.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(end) / max(done - timed_from, 1)
    t = torch.tensor([ms], device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    checksum = torch.stack([p.detach().double().sum() for p in trainer.params]).sum()
    spread = checksum.clone()
    if world > 1:                                                    # replicas must stay bit-identical
        lo, hi = checksum.clone(), checksum.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        spread = hi - lo
    else:
        spread = spread * 0
    seconds = n / args.sample_rate
    return {"model": args.model, "world_size": world, "global_batch": args.batch, "steps": done,
            "ms_per_step": float(t), "audio_seconds_per_s": args.batch * seconds / (float(t) * 1e-3),
            "cuda_graph": trainer.graph is not None, "control_net": "torch.nn" if args.stock_control_net else "kernels", "first_logged_loss": first, "last_logged_loss": last, "replica_param_spread": float(spread),
            "out_dir": str(out_dir)}


def parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--data", required=True, help="directory with signals/pitchs/loudness/mfccs .npy (or its parent with train/)")
    ap.add_argument("--model", default="decoder", choices=("decoder", "autoencoder"))
    ap.add_argument("--root", default="runs")
    ap.add_argument("--name", default="debug")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5, help="steps excluded from the ms_per_step report")
    ap.add_argument("--batch", type=int, default=16, help="GLOBAL batch (config.yaml train.batch), split over the ranks")
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--ckpt-window", type=int, default=10, help="logged losses per checkpoint comparison (the reference "
                    "compares the mean of one epoch, train.py:141-151, and resets it)")
    ap.add_argument("--scales", type=int, nargs="+", default=[4096, 2048, 1024, 512, 256, 128])
    ap.add_argument("--overlap", type=float, default=0.75)
    ap.add_argument("--hidden-size", type=int, default=512)
    ap.add_argument("--n-harmonic", type=int, default=100)
    ap.add_argument("--n-bands", type=int, default=65)
    ap.add_argument("--sample-rate", type=int, default=16000)
    ap.add_argument("--no-reverb", action="store_true")
    ap.add_argument("--cpu-noise", action="store_true", help="draw the filtered-noise excitation with the CPU generator as the reference does")
    ap.add_argument("--stock-control-net", action="store_true",
                    help="run the control net on stock torch.nn layers (cuBLAS, cuDNN) instead of this repo's kernels")
    ap.add_argument("--no-graph", action="store_true", help="run forward + backward eagerly instead of replaying a CUDA graph")
    ap.add_argument("--log-every", type=int, default=10)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--make-synthetic", type=int, default=0, metavar="N",
                    help="first write a synthetic dataset of N examples into --data (rank 0)")
    return ap


def main(argv: Optional[Sequence[str]] = None) -> None:
    args = parser().parse_args(argv)
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))))
    if args.make_synthetic:
        if rank == 0:
            write_synthetic_dataset(args.data, args.make_synthetic, args.sample_rate, seed=args.seed)
        if world > 1:
            dist.barrier()
    report = run(args)
    if rank == 0:
        print(json.dumps(report))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
