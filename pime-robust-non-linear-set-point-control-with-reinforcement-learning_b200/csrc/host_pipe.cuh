// host_pipe.cuh -- the host-buffer rollout entries (pime_wt_rollout_host_f32 / pime_ph_rollout_host_f32) as a three-stage
// pipeline over slices of the env range: while slice k runs the fused rollout on the caller's stream, slice k+1's state is
// on its way in (copy-in stream) and slice k-1's results are on their way out (copy-out stream).  PCIe is full duplex, the
// copy engines are idle while the kernel runs, and an env's random stream is keyed by its GLOBAL id (args->env_offset +
// index), so the slices produce exactly the bytes one launch over all envs produces (tests/test_gpu_03_rollout.py).
// The exposed transfer time drops from all of H2D + D2H to the first slice's H2D and the last slice's D2H.
//
// A slice is a whole number of waves (SM count x 256 envs: every persistent CTA gets the same number of tiles), at most
// kMaxSlices of them, and at least four waves long -- below 8 waves there is one slice and the entry is the plain
// copy / launch / copy sequence.  Per-step [T][n] buffers in the argument block (GPU-resident replay, injected noise) are laid
// out over the full env range: a slice gets them pre-offset with args->ld = n (shift_step_buffers).
#pragma once

#include <mutex>

#include "pime_common.cuh"
#include "tc_mlp.cuh"

namespace pime {

constexpr int kMaxSlices = 8;

struct HostArr {
    void *hp, *dp;   // host / device base pointers (either may be NULL: the array is skipped)
    int elem;        // bytes per env
    bool back;       // copied back after the rollout
};

template <typename E> inline HostArr host_arr(E *hp, E *dp, bool back) { return {hp, dp, (int)sizeof(E), back}; }

struct HostPipe {
    bool ready = false;
    cudaStream_t in = nullptr, out = nullptr;
    cudaEvent_t start = nullptr, out_done = nullptr, in_done[kMaxSlices] = {}, k_done[kMaxSlices] = {};
};

// forced slice count (tests, tuning): 0 = automatic
inline int &host_slices_override() {
    static int v = 0;
    return v;
}

inline int host_slice_count(int64_t n, bool single) {
    if (single) return 1;
    const int64_t wave = (int64_t)device_sm_count() * tc::kTileEnvs;
    int64_t c = host_slices_override() > 0 ? host_slices_override() : n / (4 * wave);
    if (c > kMaxSlices) c = kMaxSlices;
    if (c > (n + tc::kTileEnvs - 1) / tc::kTileEnvs) c = (n + tc::kTileEnvs - 1) / tc::kTileEnvs;
    return c < 1 ? 1 : (int)c;
}

inline int64_t host_slice_len(int64_t n, int slices) {
    if (slices <= 1) return n;
    const int64_t wave = (int64_t)device_sm_count() * tc::kTileEnvs;
    const int64_t unit = host_slices_override() > 0 ? tc::kTileEnvs : wave;
    const int64_t per = (n + slices - 1) / slices;
    return (per + unit - 1) / unit * unit;
}

inline std::mutex &host_pipe_mutex() {
    static std::mutex m;
    return m;
}

// the streams / events of the current device, created on first use (call with host_pipe_mutex() held)
inline int host_pipe_get(HostPipe **out) {
    static HostPipe pipes[64];
    int dev = 0;
    PIME_CUDA(cudaGetDevice(&dev));
    PIME_REQUIRE(dev >= 0 && dev < 64, "device index");
    HostPipe &p = pipes[dev];
    if (!p.ready) {
        PIME_CUDA(cudaStreamCreateWithFlags(&p.in, cudaStreamNonBlocking));
        PIME_CUDA(cudaStreamCreateWithFlags(&p.out, cudaStreamNonBlocking));
        PIME_CUDA(cudaEventCreateWithFlags(&p.start, cudaEventDisableTiming));
        PIME_CUDA(cudaEventCreateWithFlags(&p.out_done, cudaEventDisableTiming));
        for (int k = 0; k < kMaxSlices; ++k) {
            PIME_CUDA(cudaEventCreateWithFlags(&p.in_done[k], cudaEventDisableTiming));
            PIME_CUDA(cudaEventCreateWithFlags(&p.k_done[k], cudaEventDisableTiming));
        }
        p.ready = true;
    }
    *out = &p;
    return PIME_OK;
}

// the per-step buffers of a slice that starts at env `off`: S floats per replay state row, `elem` bytes per plant scalar
inline void shift_step_buffers(pime_rollout_args &a, int64_t off, int S, int elem) {
    if (a.eps) a.eps += off;
    if (a.pnoise1) a.pnoise1 = (const char *)a.pnoise1 + off * elem;
    if (a.pnoise2) a.pnoise2 = (const char *)a.pnoise2 + off * elem;
    if (a.buf_state) a.buf_state += off * S;
    if (a.buf_other) a.buf_other += off * 4;
    if (a.env_action) a.env_action = (char *)a.env_action + off * elem;
}

// launch(off, cnt, args_of_the_slice) runs the fused rollout of envs [off, off + cnt) on stream s.
template <typename Launch>
int host_pipelined_rollout(int64_t n, const HostArr *arr, int na, float *ep_dev, float *ep_host, const pime_rollout_args *args,
                           cudaStream_t s, Launch launch, bool single) {
    if (n == 0) return PIME_OK;
    const int slices = host_slice_count(n, single);
    const int64_t len = host_slice_len(n, slices);
    PIME_CUDA(cudaMemsetAsync(ep_dev, 0, (size_t)n * 4, s));
    if (slices == 1) {
        for (int j = 0; j < na; ++j)
            if (arr[j].hp && arr[j].dp) PIME_CUDA(cudaMemcpyAsync(arr[j].dp, arr[j].hp, (size_t)n * arr[j].elem, cudaMemcpyHostToDevice, s));
        if (int rc = launch((int64_t)0, n, *args)) return rc;
        if (ep_host) PIME_CUDA(cudaMemcpyAsync(ep_host, ep_dev, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        for (int j = 0; j < na; ++j)
            if (arr[j].back && arr[j].hp && arr[j].dp)
                PIME_CUDA(cudaMemcpyAsync(arr[j].hp, arr[j].dp, (size_t)n * arr[j].elem, cudaMemcpyDeviceToHost, s));
        PIME_CUDA(cudaStreamSynchronize(s));
        return PIME_OK;
    }
    std::lock_guard<std::mutex> lock(host_pipe_mutex());
    HostPipe *p = nullptr;
    if (int rc = host_pipe_get(&p)) return rc;
    PIME_CUDA(cudaEventRecord(p->start, s));               // the device arrays may still be in use by earlier work on s
    PIME_CUDA(cudaStreamWaitEvent(p->in, p->start, 0));
    int k = 0;
    for (int64_t off = 0; off < n; off += len, ++k) {
        const int64_t cnt = n - off < len ? n - off : len;
        for (int j = 0; j < na; ++j)
            if (arr[j].hp && arr[j].dp)
                PIME_CUDA(cudaMemcpyAsync((char *)arr[j].dp + off * arr[j].elem, (const char *)arr[j].hp + off * arr[j].elem,
                                          (size_t)cnt * arr[j].elem, cudaMemcpyHostToDevice, p->in));
        PIME_CUDA(cudaEventRecord(p->in_done[k], p->in));
        PIME_CUDA(cudaStreamWaitEvent(s, p->in_done[k], 0));
        pime_rollout_args a = *args;
        a.env_offset = args->env_offset + (uint64_t)off;
        a.ld = args->ld ? args->ld : n;
        if (int rc = launch(off, cnt, a)) {
            cudaStreamSynchronize(p->in);
            cudaStreamSynchronize(p->out);
            return rc;
        }
        PIME_CUDA(cudaEventRecord(p->k_done[k], s));
        PIME_CUDA(cudaStreamWaitEvent(p->out, p->k_done[k], 0));
        if (ep_host) PIME_CUDA(cudaMemcpyAsync(ep_host + off, ep_dev + off, (size_t)cnt * 4, cudaMemcpyDeviceToHost, p->out));
        for (int j = 0; j < na; ++j)
            if (arr[j].back && arr[j].hp && arr[j].dp)
                PIME_CUDA(cudaMemcpyAsync((char *)arr[j].hp + off * arr[j].elem, (const char *)arr[j].dp + off * arr[j].elem,
                                          (size_t)cnt * arr[j].elem, cudaMemcpyDeviceToHost, p->out));
    }
    PIME_CUDA(cudaEventRecord(p->out_done, p->out));
    PIME_CUDA(cudaStreamWaitEvent(s, p->out_done, 0));     // later work on s sees the call as complete
    PIME_CUDA(cudaStreamSynchronize(s));
    return PIME_OK;
}

}  // namespace pime
