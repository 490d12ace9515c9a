// Host-buffer entry points: a (pinned) host trajectory is streamed to the device in chunks on two
// private streams, each chunk's H2D copy overlapping the evaluation of the previous one
// (Trajectory.get_raman_spectrum on a numpy trajectory, ramannoodle/dynamics/_trajectory.py:71-90).
//
// Stream order.  The private streams first wait on an event recorded on the caller's stream, so work
// the caller enqueued before the call (a cross-rank barrier, a consumer of the previous contents of the
// output buffers) is complete before the first copy or kernel; the calls return after both private
// streams have drained.
#include "rn_common.cuh"

namespace rn {

struct HostPipe {
    double* d_pos[2] = {nullptr, nullptr};
    double* d_alpha[2] = {nullptr, nullptr};
    cudaStream_t stream[2] = {nullptr, nullptr};
    cudaEvent_t entry = nullptr;
    void release() {
        for (int i = 0; i < 2; i++) {
            if (d_pos[i]) cudaFree(d_pos[i]);
            if (d_alpha[i]) cudaFree(d_alpha[i]);
            if (stream[i]) cudaStreamDestroy(stream[i]);
            d_pos[i] = d_alpha[i] = nullptr;
            stream[i] = nullptr;
        }
        if (entry) cudaEventDestroy(entry);
        entry = nullptr;
    }
    // no destructor: at process exit the CUDA context may already be gone
};

// Staging buffers and streams, cached per thread (allocation / free would serialise the device).
static int acquire_pipe(int device, int64_t pos_doubles, int64_t alpha_doubles, HostPipe** out) {
    static thread_local HostPipe pipe;
    static thread_local int pipe_device = -1;
    static thread_local int64_t pipe_pos_doubles = 0, pipe_alpha_doubles = 0;
    if (pipe_device != device) {
        pipe.release();
        pipe_device = device;
        pipe_pos_doubles = pipe_alpha_doubles = 0;
        for (int i = 0; i < 2; i++) RN_CUDA(cudaStreamCreateWithFlags(&pipe.stream[i], cudaStreamNonBlocking));
        RN_CUDA(cudaEventCreateWithFlags(&pipe.entry, cudaEventDisableTiming));
    }
    if (pipe_pos_doubles < pos_doubles) {
        for (int i = 0; i < 2; i++) {
            if (pipe.d_pos[i]) RN_CUDA(cudaFree(pipe.d_pos[i]));
            pipe.d_pos[i] = nullptr;
            RN_CUDA(cudaMalloc((void**)&pipe.d_pos[i], sizeof(double) * pos_doubles));
        }
        pipe_pos_doubles = pos_doubles;
    }
    if (pipe_alpha_doubles < alpha_doubles) {
        for (int i = 0; i < 2; i++) {
            if (pipe.d_alpha[i]) RN_CUDA(cudaFree(pipe.d_alpha[i]));
            pipe.d_alpha[i] = nullptr;
            RN_CUDA(cudaMalloc((void**)&pipe.d_alpha[i], sizeof(double) * alpha_doubles));
        }
        pipe_alpha_doubles = alpha_doubles;
    }
    *out = &pipe;
    return RN_OK;
}

// private streams start after everything already enqueued on the caller's stream
static int order_after_caller(HostPipe& pipe, cudaStream_t caller) {
    RN_CUDA(cudaEventRecord(pipe.entry, caller));
    for (int i = 0; i < 2; i++) RN_CUDA(cudaStreamWaitEvent(pipe.stream[i], pipe.entry, 0));
    return RN_OK;
}

static int64_t pick_chunk(int64_t chunk_frames, int64_t num_frames, int64_t K) {
    // ~256 MiB chunks: measured on B200 (tools/e2e_probe2.py) 64 MiB chunks show sporadic multi-100-ms
    // stalls, 256 MiB chunks run at a steady ~48 GB/s of the 55 GB/s pinned-copy rate
    if (chunk_frames <= 0) chunk_frames = std::max<int64_t>(8, (int64_t)(256ll << 20) / (K * 8));
    chunk_frames = std::min(chunk_frames, num_frames);
    return (chunk_frames + 7) / 8 * 8;
}

}  // namespace rn

using namespace rn;

extern "C" int rn_host_register(void* h_ptr, size_t bytes) {
    RN_CHECK_ARG(h_ptr != nullptr && bytes > 0, "invalid host buffer");
    RN_CUDA(cudaHostRegister(h_ptr, bytes, cudaHostRegisterDefault));
    return RN_OK;
}

extern "C" int rn_host_unregister(void* h_ptr) {
    RN_CHECK_ARG(h_ptr != nullptr, "invalid host buffer");
    RN_CUDA(cudaHostUnregister(h_ptr));
    return RN_OK;
}

// The chunk loop of every host entry: chunk [f0, f0 + n) is copied into staging slot `slot` on that slot's
// stream and evaluated there by step(d_pos, out, f0, n, stream) -> rn_status, so that the copy of one chunk
// overlaps the evaluation of the other.  `out` is where the chunk's rows go: d_alpha + 9 f0, a staging buffer
// when only h_alpha is given, null when neither is (a sweep stores to its own outputs); h_alpha receives the
// rows of every chunk.
template <class Step>
static int host_chunks(int device, int64_t K, const double* h_positions, int64_t num_frames, int64_t chunk_frames,
                       double* h_alpha, double* d_alpha, void* stream, Step step) {
    DeviceGuard guard(device);
    if (!guard.ok) {
        set_error("cudaSetDevice(%d) failed", device);
        return RN_ERR_CUDA;
    }
    chunk_frames = pick_chunk(chunk_frames, num_frames, K);
    const bool stage_alpha = h_alpha && !d_alpha;
    HostPipe* pipe = nullptr;
    int rc = acquire_pipe(device, chunk_frames * K, stage_alpha ? chunk_frames * 9 : 0, &pipe);
    if (rc != RN_OK) return rc;
    rc = order_after_caller(*pipe, static_cast<cudaStream_t>(stream));
    if (rc != RN_OK) return rc;
    int slot = 0;
    for (int64_t f0 = 0; f0 < num_frames; f0 += chunk_frames, slot ^= 1) {
        const int64_t n = std::min(chunk_frames, num_frames - f0);
        cudaStream_t s = pipe->stream[slot];
        // stream order serialises reuse of this slot's buffers; the other slot overlaps
        RN_CUDA(cudaMemcpyAsync(pipe->d_pos[slot], h_positions + f0 * K, sizeof(double) * n * K, cudaMemcpyHostToDevice, s));
        double* out = d_alpha ? d_alpha + f0 * 9 : stage_alpha ? pipe->d_alpha[slot] : nullptr;
        rc = step(pipe->d_pos[slot], out, f0, n, s);
        if (rc != RN_OK) return rc;
        if (h_alpha) RN_CUDA(cudaMemcpyAsync(h_alpha + f0 * 9, out, sizeof(double) * n * 9, cudaMemcpyDeviceToHost, s));
    }
    RN_CUDA(cudaStreamSynchronize(pipe->stream[0]));
    RN_CUDA(cudaStreamSynchronize(pipe->stream[1]));
    return RN_OK;
}

// One model: d_alpha is the local series (or null when only h_alpha is wanted); `peers` describes further
// destinations of the rows (broadcast or routed, rn_common.cuh).
static int host_pipeline(const rn_model* model, const double* h_positions, int64_t num_frames, double* h_alpha,
                         double* d_alpha, const AlphaPeers& peers, int64_t chunk_frames, void* stream) {
    RN_CHECK_ARG(model != nullptr, "model is null");
    RN_CHECK_ARG(num_frames >= 0, "num_frames must be non-negative");
    if (num_frames == 0) return RN_OK;
    RN_CHECK_ARG(h_positions != nullptr, "null host pointer");
    RN_CHECK_ARG(h_alpha || d_alpha, "no output buffer given");
    return host_chunks(model->device, model->dim, h_positions, num_frames, chunk_frames, h_alpha, d_alpha, stream,
                       [&](const double* d_pos, double* out, int64_t f0, int64_t n, cudaStream_t s) {
                           return eval_with_peers(model, d_pos, n, out, s, peers_at(peers, f0));
                       });
}

extern "C" int rn_calc_polarizabilities_host(const rn_model* model, const double* h_positions, int64_t num_frames,
                                             double* h_alpha, double* d_alpha, int64_t chunk_frames) {
    return host_pipeline(model, h_positions, num_frames, h_alpha, d_alpha, no_peers(), chunk_frames, nullptr);
}

extern "C" int rn_calc_polarizabilities_host_multi(const rn_model* model, const double* h_positions, int64_t num_frames,
                                                   double* const* d_alpha_outputs, int num_outputs,
                                                   int64_t chunk_frames, void* stream) {
    RN_CHECK_ARG(d_alpha_outputs != nullptr && num_outputs >= 1 && num_outputs <= 8,
                 "between 1 and 8 output pointers are required");
    for (int i = 0; i < num_outputs; i++) RN_CHECK_ARG(d_alpha_outputs[i] != nullptr, "null output pointer");
    AlphaPeers peers = no_peers();
    peers.count = num_outputs - 1;
    for (int i = 1; i < num_outputs; i++) peers.ptr[i - 1] = d_alpha_outputs[i];
    return host_pipeline(model, h_positions, num_frames, nullptr, d_alpha_outputs[0], peers, chunk_frames, stream);
}

extern "C" int rn_calc_polarizabilities_host_routed(const rn_model* model, const double* h_positions,
                                                    int64_t num_frames, double* d_alpha, double* const* peer_series,
                                                    int world, int64_t first_frame, int64_t period, int64_t width,
                                                    int64_t chunk_frames, void* stream) {
    AlphaPeers peers;
    int rc = make_routed_peers(peer_series, world, first_frame, period, width, &peers);
    if (rc != RN_OK) return rc;
    RN_CHECK_ARG(d_alpha != nullptr, "null output pointer");
    return host_pipeline(model, h_positions, num_frames, nullptr, d_alpha, peers, chunk_frames, stream);
}

// Mask sweep from a host trajectory: every chunk crosses PCIe once and is evaluated by all models.  `routed`
// (null, or one entry per model) names the ranks the rows also go to.
static int host_sweep(const rn_model* const* models, int num_models, const double* h_positions, int64_t num_frames,
                      double* const* d_alpha_outputs, const AlphaPeers* routed, int64_t chunk_frames, void* stream) {
    RN_CHECK_ARG(models != nullptr && num_models >= 1 && num_models <= kMaxSweepModels, "1..64 models are required");
    RN_CHECK_ARG(d_alpha_outputs != nullptr, "output pointers are required");
    for (int g = 0; g < num_models; g++) {
        RN_CHECK_ARG(models[g] != nullptr && d_alpha_outputs[g] != nullptr, "null model or output pointer");
        RN_CHECK_ARG(models[g]->device == models[0]->device && models[g]->dim == models[0]->dim,
                     "models of a sweep must live on one device and describe the same structure");
    }
    RN_CHECK_ARG(num_frames >= 0, "num_frames must be non-negative");
    if (num_frames == 0) return RN_OK;
    RN_CHECK_ARG(h_positions != nullptr, "null host pointer");
    return host_chunks(models[0]->device, models[0]->dim, h_positions, num_frames, chunk_frames, nullptr, nullptr,
                       stream, [&](const double* d_pos, double*, int64_t f0, int64_t n, cudaStream_t s) {
                           double* outs[kMaxSweepModels];
                           AlphaPeers chunk_routed[kMaxSweepModels];
                           for (int g = 0; g < num_models; g++) {
                               outs[g] = d_alpha_outputs[g] + f0 * 9;
                               if (routed) chunk_routed[g] = peers_at(routed[g], f0);
                           }
                           return sweep_eval(models, num_models, d_pos, n, outs, s, routed ? chunk_routed : nullptr);
                       });
}

extern "C" int rn_calc_polarizabilities_host_sweep(const rn_model* const* models, int num_models,
                                                   const double* h_positions, int64_t num_frames,
                                                   double* const* d_alpha_outputs, int64_t chunk_frames) {
    return host_sweep(models, num_models, h_positions, num_frames, d_alpha_outputs, nullptr, chunk_frames, nullptr);
}

extern "C" int rn_calc_polarizabilities_host_sweep_routed(const rn_model* const* models, int num_models,
                                                          const double* h_positions, int64_t num_frames,
                                                          double* const* d_alpha_outputs, double* const* peer_series,
                                                          int world, int64_t first_frame, int64_t period, int64_t width,
                                                          int64_t chunk_frames, void* stream) {
    AlphaPeers routed[kMaxSweepModels];
    const int rc = make_sweep_peers(num_models, peer_series, world, first_frame, period, width, routed);
    if (rc != RN_OK) return rc;
    return host_sweep(models, num_models, h_positions, num_frames, d_alpha_outputs, routed, chunk_frames, stream);
}
