"""Config 3 (realtime export path): per-buffer latency of the scripted model, measured the way the Pd
external calls it (ddsp_model.cpp:32-51): 1024 host floats of pitch and loudness -> device -> forward ->
host.  48 kHz, block 512, 64 harmonics, 65 bands, hidden 512, batch 1.  First line: the dry export (reverb left
to the host); second line: the same model exported with streaming_reverb=True (the trained 48000-tap reverb,
its tail carried across buffers), and the latency it adds.  The two exports are called alternately.
Budget per buffer: 1024/48000 = 21.3 ms."""
import json, os, sys, time, tempfile
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ddsp_pytorch_b200  # noqa
from ddsp_pytorch_b200.models.decoder import DDSPDecoder
from ddsp_pytorch_b200.export import export_torchscript

torch.manual_seed(0)
model = DDSPDecoder(hidden_size=512, n_harmonic=64, n_bands=65, sample_rate=48000, block_size=512, has_reverb=True)
model = model.cuda().eval()
tmp = tempfile.mkdtemp()
export_torchscript(model, os.path.join(tmp, "rt.ts"), mean_loudness=-30.0, std_loudness=10.0, realtime=True)
export_torchscript(model, os.path.join(tmp, "rt_reverb.ts"), mean_loudness=-30.0, std_loudness=10.0, realtime=True,
                   streaming_reverb=True)
modules = {"dry": torch.jit.load(os.path.join(tmp, "rt.ts")).cuda(),
           "reverb": torch.jit.load(os.path.join(tmp, "rt_reverb.ts")).cuda()}
pitch = torch.full((1, 1024, 1), 220.0).pin_memory()
loud = torch.full((1, 1024, 1), -25.0).pin_memory()
out_host = torch.empty(1, 1024, 1).pin_memory()
def call(rt):
    with torch.no_grad():
        y = rt(pitch.cuda(non_blocking=True), loud.cuda(non_blocking=True))
        out_host.copy_(y, non_blocking=True)
        torch.cuda.synchronize()
for _ in range(30):
    for rt in modules.values():
        call(rt)
ts = {k: [] for k in modules}
for _ in range(300):
    for k, rt in modules.items():
        t0 = time.perf_counter(); call(rt); ts[k].append((time.perf_counter() - t0) * 1e3)
for v in ts.values():
    v.sort()
med = {k: v[len(v) // 2] for k, v in ts.items()}
p99 = {k: v[int(len(v) * 0.99)] for k, v in ts.items()}
budget = 1024 / 48000 * 1e3
print(json.dumps({"config": "configs[2] realtime export: 48 kHz, block 512, 64 harmonics, batch 1, 1024-sample buffers",
                  "ms_per_buffer_median": med["dry"], "ms_per_buffer_p99": p99["dry"],
                  "budget_ms": budget, "realtime_factor": budget / med["dry"],
                  "includes": "H2D of 2x1024 floats, control net (cluster GRU kernel, library GEMMs at this size), synth kernels, D2H of 1024 floats"}))
print(json.dumps({"config": "the same export with streaming_reverb=True: 48000-tap reverb, history carried across buffers",
                  "ms_per_buffer_median": med["reverb"], "ms_per_buffer_p99": p99["reverb"],
                  "budget_ms": budget, "realtime_factor": budget / med["reverb"],
                  "added_ms_median": med["reverb"] - med["dry"], "added_ms_p99": p99["reverb"] - p99["dry"],
                  "includes": "the dry line's work + impulse build, conv_stream (two launches), history copy"}))
