// Link-level check of the drop-in boundary: this translation unit uses the warp-transducer API (rnnt.h) through this
// project's drop-in header include/rnnt_b200.h and is linked against librnnt_b200.so.  It is what a binding such as
// tensorflow_binding/src/warprnnt_op.cc:105-141 or pytorch_binding/src/binding.cpp:84-154 does with the library:
// get_workspace_size -> device workspace -> compute_rnnt_loss(RNNT_GPU, device labels/lengths, HOST costs) -> status
// string.  Built with -DRNNT_REFERENCE_HEADER it includes the reference's own rnnt.h instead (found through -I, never
// copied into this repo): tests/golden/make_golden.py does so to record the reference header's layout, which
// tests/test_abi.py holds this header's layout to.
// Data: the reference's own known-answer test (tests/test_cpu.cpp:12-71 / test_gpu.cu small_test): B=1 T=2 U=3 V=5,
// expected cost 4.495666 and the logits gradient of pytorch_binding/test/test.py:62-74.
// Modes:  abi_harness layout -> prints the rnntOptions layout and the enum values as one JSON line
//         abi_harness link   -> resolves every symbol and checks the host-only entry points (no GPU needed)
//         abi_harness run    -> runs the KAT on cuda:0
#ifdef RNNT_REFERENCE_HEADER
#include <rnnt.h>
#else
#include <rnnt_b200.h>
#endif

#include <cuda_runtime.h>

#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <vector>

static int fail(const char* what) { std::fprintf(stderr, "abi_harness: FAILED: %s\n", what); return 1; }

static void print_layout() {
    std::printf("{\"sizeof_rnntOptions\": %zu, \"offsets\": {\"loc\": %zu, \"num_threads\": %zu, \"stream\": %zu, "
                "\"blank_label\": %zu, \"maxT\": %zu, \"maxU\": %zu, \"batch_first\": %zu}, "
                "\"status\": [%d, %d, %d, %d, %d], \"location\": [%d, %d]}\n",
                sizeof(rnntOptions), offsetof(rnntOptions, loc), offsetof(rnntOptions, num_threads),
                offsetof(rnntOptions, stream), offsetof(rnntOptions, blank_label), offsetof(rnntOptions, maxT),
                offsetof(rnntOptions, maxU), offsetof(rnntOptions, batch_first),
                (int)RNNT_STATUS_SUCCESS, (int)RNNT_STATUS_MEMOPS_FAILED, (int)RNNT_STATUS_INVALID_VALUE,
                (int)RNNT_STATUS_EXECUTION_FAILED, (int)RNNT_STATUS_UNKNOWN_ERROR, (int)RNNT_CPU, (int)RNNT_GPU);
}

int main(int argc, char** argv) {
    if (argc > 1 && !std::strcmp(argv[1], "layout")) { print_layout(); return 0; }
    const bool run = argc > 1 && !std::strcmp(argv[1], "run");
    if (get_warprnnt_version() != 1) return fail("get_warprnnt_version");
    if (std::strcmp(rnntGetStatusString(RNNT_STATUS_SUCCESS), "no error")) return fail("status string");
    if (std::strcmp(rnntGetStatusString(RNNT_STATUS_INVALID_VALUE), "invalid value")) return fail("status string 2");
    static_assert(sizeof(rnntOptions) == 32, "rnntOptions is a 32-byte by-value struct on x86-64");
    const int B = 1, T = 2, U = 3, V = 5;
    size_t ws_bytes = 0;
    if (get_workspace_size(T, U, B, true, &ws_bytes) != RNNT_STATUS_SUCCESS || ws_bytes == 0) return fail("get_workspace_size");
    if (get_workspace_size(0, U, B, true, &ws_bytes) != RNNT_STATUS_INVALID_VALUE) return fail("get_workspace_size argument check");
    rnntOptions opt{};
    opt.loc = RNNT_GPU; opt.num_threads = 0; opt.stream = nullptr; opt.blank_label = 0; opt.maxT = T; opt.maxU = U; opt.batch_first = true;
    float cost = 0.f;
    if (compute_rnnt_loss(nullptr, nullptr, nullptr, nullptr, nullptr, V, B, &cost, nullptr, opt) != RNNT_STATUS_INVALID_VALUE)
        return fail("compute_rnnt_loss argument check");
    // the address of the fp64 twin is taken so that the linker must resolve it as well
    auto f64 = &compute_rnnt_loss_fp64;
    if (!f64) return fail("compute_rnnt_loss_fp64");
    if (!run) { std::printf("abi_harness: link ok (%zu workspace bytes for the KAT)\n", ws_bytes); return 0; }

    const float acts[B * T * U * V] = {0.1f, 0.6f, 0.1f, 0.1f, 0.1f, 0.1f, 0.1f, 0.6f, 0.1f, 0.1f, 0.1f, 0.1f, 0.2f, 0.8f, 0.1f,
                                       0.1f, 0.6f, 0.1f, 0.1f, 0.1f, 0.1f, 0.1f, 0.2f, 0.1f, 0.1f, 0.7f, 0.1f, 0.2f, 0.1f, 0.1f};
    const int labels[2] = {1, 2}, ylen[1] = {2}, xlen[1] = {T};
    float *d_acts, *d_grads; int *d_lab, *d_ylen, *d_xlen; void* d_ws;
    if (cudaMalloc(&d_acts, sizeof(acts)) || cudaMalloc(&d_grads, sizeof(acts)) || cudaMalloc(&d_lab, sizeof(labels)) ||
        cudaMalloc(&d_ylen, 4) || cudaMalloc(&d_xlen, 4) || cudaMalloc(&d_ws, ws_bytes)) return fail("cudaMalloc");
    cudaMemcpy(d_acts, acts, sizeof(acts), cudaMemcpyHostToDevice);
    cudaMemcpy(d_lab, labels, sizeof(labels), cudaMemcpyHostToDevice);
    cudaMemcpy(d_ylen, ylen, 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_xlen, xlen, 4, cudaMemcpyHostToDevice);
    const rnntStatus_t st = compute_rnnt_loss(d_acts, d_grads, d_lab, d_ylen, d_xlen, V, B, &cost, d_ws, opt);
    if (st != RNNT_STATUS_SUCCESS) { std::fprintf(stderr, "status: %s\n", rnntGetStatusString(st)); return fail("compute_rnnt_loss"); }
    std::vector<float> g(B * T * U * V);
    cudaMemcpy(g.data(), d_grads, sizeof(acts), cudaMemcpyDeviceToHost);
    const float want_first_row[5] = {-0.13116688f, -0.3999269f, 0.17703125f, 0.17703125f, 0.17703125f};
    if (std::fabs(cost - 4.495666f) > 1e-4f) { std::fprintf(stderr, "cost %f\n", cost); return fail("KAT cost"); }
    for (int i = 0; i < 5; ++i)
        if (std::fabs(g[i] - want_first_row[i]) > 1e-5f) { std::fprintf(stderr, "grad[%d] %f\n", i, g[i]); return fail("KAT gradient"); }
    std::printf("abi_harness: run ok, cost %.6f\n", cost);
    return 0;
}
