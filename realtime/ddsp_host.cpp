// C++ host of the exported model on CUDA: the consumer side of the drop-in boundary (SURVEY 8b, 8f-2).
//
// This is what realtime/ddsp_tilde/ddsp_model.cpp of the reference does (load a TorchScript file, then
// per audio buffer: host floats -> tensor -> forward -> host floats), with the two changes the B200 op
// library needs: the ops are registered by dlopen()-ing libddsp_b200_torch.so BEFORE torch::jit::load
// (ddsp_model.cpp:17), and the device is CUDA (ddsp_model.h:6).  No Pd dependency: `main` streams
// synthetic 1024-sample buffers the way ddsp_tilde.cpp:81-92 does (a fresh std::thread per buffer) and
// prints a checksum and the per-buffer latency, so the path can be exercised from a test.
// All streaming state (GRU cache, oscillator phase and, in a streaming_reverb export, the reverb's history) lives
// in the module's buffers: the same host plays a dry export and one that convolves its own reverb.
//
//   ddsp_host <libddsp_b200_torch.so> <model.ts> [buffers=8] [buffer_size=1024]
#include <torch/script.h>
#include <torch/torch.h>

#include <dlfcn.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

class DDSPModelCuda {
public:
    int load(const std::string &ops_library, const std::string &path) {
        if (!dlopen(ops_library.c_str(), RTLD_NOW | RTLD_GLOBAL)) {       // registers ddsp_b200::* ops
            std::fprintf(stderr, "dlopen failed: %s\n", dlerror());
            return 1;
        }
        try {
            module_ = torch::jit::load(path, torch::kCUDA);
            module_.eval();
            loaded_ = true;
            return 0;
        } catch (const std::exception &e) {
            std::fprintf(stderr, "%s\n", e.what());
            return 1;
        }
    }

    // same contract as DDSPModel::perform (ddsp_model.cpp:32-51)
    void perform(float *pitch, float *loudness, float *out_buffer, int buffer_size) {
        torch::NoGradGuard no_grad;
        if (!loaded_) return;
        auto p = torch::from_blob(pitch, {1, buffer_size, 1}).to(torch::kCUDA);
        auto l = torch::from_blob(loudness, {1, buffer_size, 1}).to(torch::kCUDA);
        std::vector<torch::jit::IValue> inputs = {p, l};
        auto out = module_.forward(inputs).toTensor().to(torch::kCPU).contiguous();
        std::memcpy(out_buffer, out.data_ptr<float>(), buffer_size * sizeof(float));
    }

private:
    torch::jit::script::Module module_;
    bool loaded_ = false;
};

int main(int argc, char **argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: %s <libddsp_b200_torch.so> <model.ts> [buffers] [buffer_size]\n", argv[0]);
        return 2;
    }
    const int buffers = argc > 3 ? std::atoi(argv[3]) : 8;
    const int n = argc > 4 ? std::atoi(argv[4]) : 1024;
    DDSPModelCuda model;
    if (model.load(argv[1], argv[2])) return 1;

    std::vector<float> pitch(n), loud(n), out(n);
    double checksum = 0.0, peak = 0.0, worst_ms = 0.0, total_ms = 0.0;
    float prev_last = 0.f, max_jump = 0.f;
    for (int b = 0; b < buffers + 2; ++b) {
        for (int i = 0; i < n; ++i) {
            pitch[i] = 220.0f + 20.0f * std::sin(0.001f * (float)(b * n + i));
            loud[i] = -25.0f;
        }
        const auto t0 = std::chrono::steady_clock::now();
        std::thread worker([&] { model.perform(pitch.data(), loud.data(), out.data(), n); });   // ddsp_tilde.cpp:88
        worker.join();
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (b >= 2) {                                  // first calls pay CUDA / cuDNN initialisation
            total_ms += ms;
            worst_ms = ms > worst_ms ? ms : worst_ms;
        }
        for (int i = 0; i < n; ++i) {
            if (!std::isfinite(out[i])) { std::fprintf(stderr, "non-finite output\n"); return 1; }
            checksum += out[i];
            peak = std::fabs(out[i]) > peak ? std::fabs(out[i]) : peak;
        }
        if (b > 0) max_jump = std::fabs(out[0] - prev_last) > max_jump ? std::fabs(out[0] - prev_last) : max_jump;
        prev_last = out[n - 1];
    }
    std::printf("{\"buffers\": %d, \"buffer_size\": %d, \"checksum\": %.6f, \"peak\": %.6f, \"boundary_jump\": %.6f, "
                "\"mean_ms\": %.4f, \"worst_ms\": %.4f}\n",
                buffers, n, checksum, peak, max_jump, total_ms / buffers, worst_ms);
    return 0;
}
