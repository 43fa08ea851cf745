// vx_multi.cu -- one process per GPU: peer-mapped buffers (CUDA IPC) and the cross-GPU hand-off flags the stripe
// composite is built on.
//
// The reference hands every Rayon worker a disjoint `&mut` stripe of ONE framebuffer (framebuffer.rs:392-431,
// main.rs:581-597).  The B200 form of that: the composed frame lives in GPU0's HBM, every other GPU maps it through
// CUDA IPC and its raster kernel's write-out stores the stripe straight over NVLink (vx_render_frame_into with the
// mapped pointer) -- no staging buffer, no collective.  What is left to exchange per frame is one 32-bit counter per
// rank:
//   vx_signal_flags   enqueued behind the raster kernel: fence at system scope, then store the frame number into the
//                     composing GPU's flag word (peer store)
//   vx_wait_flags     enqueued on the composing GPU: one warp polls its LOCAL flag words (L2 hits) until every rank
//                     has published that frame number; bounded by a timeout so a lost peer cannot hang the device
// and the same pair in the other direction as the "frame consumed, buffer free" acknowledgement.
#include "vx_common.cuh"

namespace {

__global__ void signal_flags_kernel(uint32_t *const *flags, int n, uint32_t value) {
    // the preceding kernels of this stream have completed (stream order); make their peer stores visible system-wide
    // before the flag that announces them
    __threadfence_system();
    const int i = threadIdx.x;
    if (i < n && flags[i]) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flags[i]), "r"(value) : "memory");
}

__global__ void signal_flag_kernel(uint32_t *flag, uint32_t value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}

// status[0] = 0 ok / 1 timed out; status[1] = the lowest flag value seen at the end
__global__ void wait_flags_kernel(const uint32_t *flags, int n, int stride_words, uint32_t value, unsigned long long timeout_ns, uint32_t *status) {
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    const int lane = threadIdx.x;
    bool timed_out = false;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        while (true) {
            uint32_t v = value;
            if (i < n) asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + (size_t)i * stride_words) : "memory");
            // frame numbers wrap: "reached" = not more than 2^31 behind
            const bool ok = (int32_t)(v - value) >= 0;
            if (__all_sync(0xffffffffu, ok)) break;
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > timeout_ns) {
                timed_out = true;
                break;
            }
            __nanosleep(40);
        }
        if (timed_out) break;
    }
    __threadfence_system();
    if (lane == 0 && status) {
        if (timed_out) status[0] = 1u;
    }
}

// wait for n_wait local flag words, then publish `sv` into n_signal flag words (one warp)
__global__ void wait_then_signal_kernel(const uint32_t *flags, int n, int stride_words, uint32_t value, unsigned long long timeout_ns, uint32_t *status,
                                        uint32_t *const *sig, int n_sig, uint32_t sv) {
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    const int lane = threadIdx.x;
    bool timed_out = false;
    for (int base = 0; base < n && !timed_out; base += 32) {
        const int i = base + lane;
        while (true) {
            uint32_t v = value;
            if (i < n) asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + (size_t)i * stride_words) : "memory");
            if (__all_sync(0xffffffffu, (int32_t)(v - value) >= 0)) break;
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > timeout_ns) {
                timed_out = true;
                break;
            }
            __nanosleep(40);
        }
    }
    __threadfence_system();
    if (timed_out) {
        if (lane == 0 && status) status[0] = 1u;
        return; // nothing is acknowledged for a frame that never arrived
    }
    if (lane < n_sig && sig[lane]) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(sig[lane]), "r"(sv) : "memory");
}

} // namespace

int vx_stage_flag_table(VxContext *ctx, uint32_t *const *flags, int n) {
    VX_CUDA(ctx, ctx->multi_ptrs.reserve(sizeof(uint32_t *) * 32));
    if (n > 0 && (ctx->multi_ptrs_n != n || memcmp(ctx->multi_ptrs_host, flags, sizeof(uint32_t *) * (size_t)n) != 0)) {
        VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // an earlier kernel may still read the table
        memcpy(ctx->multi_ptrs_host, flags, sizeof(uint32_t *) * (size_t)n);
        ctx->multi_ptrs_n = n;
        VX_CUDA(ctx, cudaMemcpyAsync(ctx->multi_ptrs.ptr, ctx->multi_ptrs_host, sizeof(uint32_t *) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    }
    return VX_OK;
}

extern "C" {

int vx_device_alloc(VxContext *ctx, size_t bytes, void **d_out) {
    if (!ctx || !d_out) return vx_fail(ctx, VX_ERR_INVALID, "vx_device_alloc: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    *d_out = nullptr;
    VX_CUDA(ctx, cudaMalloc(d_out, bytes ? bytes : 1)); // its own allocation: exportable through CUDA IPC
    VX_CUDA(ctx, cudaMemsetAsync(*d_out, 0, bytes ? bytes : 1, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return VX_OK;
}

int vx_device_free(VxContext *ctx, void *d_ptr) {
    if (!ctx) return VX_ERR_INVALID;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    if (d_ptr) VX_CUDA(ctx, cudaFree(d_ptr));
    return VX_OK;
}

int vx_ipc_export(VxContext *ctx, void *d_ptr, uint8_t handle_out[64]) {
    if (!ctx || !d_ptr || !handle_out) return vx_fail(ctx, VX_ERR_INVALID, "vx_ipc_export: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    VX_CUDA(ctx, cudaIpcGetMemHandle(&h, d_ptr));
    memcpy(handle_out, &h, 64);
    return VX_OK;
}

int vx_ipc_open(VxContext *ctx, const uint8_t handle[64], void **d_out) {
    if (!ctx || !handle || !d_out) return vx_fail(ctx, VX_ERR_INVALID, "vx_ipc_open: bad argument");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    *d_out = nullptr;
    VX_CUDA(ctx, cudaIpcOpenMemHandle(d_out, h, cudaIpcMemLazyEnablePeerAccess)); // maps the peer allocation; enables P2P over NVLink
    return VX_OK;
}

int vx_ipc_close(VxContext *ctx, void *d_ptr) {
    if (!ctx) return VX_ERR_INVALID;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    if (d_ptr) VX_CUDA(ctx, cudaIpcCloseMemHandle(d_ptr));
    return VX_OK;
}

int vx_signal_flags(VxContext *ctx, uint32_t *const *d_flags, int32_t n, uint32_t value) {
    if (!ctx || n < 0 || n > 32 || (n > 0 && !d_flags)) return vx_fail(ctx, VX_ERR_INVALID, "vx_signal_flags: bad argument (at most 32 flags)");
    if (n == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    if (n == 1) {
        signal_flag_kernel<<<1, 1, 0, ctx->stream>>>(d_flags[0], value);
        VX_CHECK_LAUNCH(ctx);
        return VX_OK;
    }
    const int rc = vx_stage_flag_table(ctx, d_flags, n);
    if (rc != VX_OK) return rc;
    signal_flags_kernel<<<1, 32, 0, ctx->stream>>>(ctx->multi_ptrs.as<uint32_t *>(), n, value);
    VX_CHECK_LAUNCH(ctx);
    return VX_OK;
}

int vx_wait_flags(VxContext *ctx, const uint32_t *d_flags, int32_t n, int32_t stride_words, uint32_t value, int32_t timeout_us) {
    if (!ctx || n < 0 || (n > 0 && !d_flags) || stride_words < 1) return vx_fail(ctx, VX_ERR_INVALID, "vx_wait_flags: bad argument");
    if (n == 0) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->multi_status.ptr) {
        VX_CUDA(ctx, ctx->multi_status.reserve(16));
        VX_CUDA(ctx, cudaMemsetAsync(ctx->multi_status.ptr, 0, 16, ctx->stream));
    }
    wait_flags_kernel<<<1, 32, 0, ctx->stream>>>(d_flags, n, stride_words, value, vx_timeout_ns(timeout_us), ctx->multi_status.as<uint32_t>());
    VX_CHECK_LAUNCH(ctx);
    return VX_OK;
}

int vx_wait_then_signal(VxContext *ctx, const uint32_t *d_wait_flags, int32_t n_wait, int32_t stride_words, uint32_t wait_value,
                        uint32_t *const *d_signal_flags, int32_t n_signal, uint32_t signal_value, int32_t timeout_us) {
    if (!ctx || n_wait < 0 || (n_wait > 0 && !d_wait_flags) || stride_words < 1 || n_signal < 0 || n_signal > 32 || (n_signal > 0 && !d_signal_flags))
        return vx_fail(ctx, VX_ERR_INVALID, "vx_wait_then_signal: bad argument (at most 32 flags to signal)");
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->multi_status.ptr) {
        VX_CUDA(ctx, ctx->multi_status.reserve(16));
        VX_CUDA(ctx, cudaMemsetAsync(ctx->multi_status.ptr, 0, 16, ctx->stream));
    }
    const int rc = vx_stage_flag_table(ctx, d_signal_flags, n_signal);
    if (rc != VX_OK) return rc;
    wait_then_signal_kernel<<<1, 32, 0, ctx->stream>>>(d_wait_flags, n_wait, stride_words, wait_value, vx_timeout_ns(timeout_us), ctx->multi_status.as<uint32_t>(),
                                                       ctx->multi_ptrs.as<uint32_t *>(), n_signal, signal_value);
    VX_CHECK_LAUNCH(ctx);
    return VX_OK;
}

int vx_wait_status(VxContext *ctx, int32_t *timed_out) {
    if (!ctx || !timed_out) return vx_fail(ctx, VX_ERR_INVALID, "vx_wait_status: bad argument");
    *timed_out = 0;
    if (!ctx->multi_status.ptr) return VX_OK;
    VX_CUDA(ctx, cudaSetDevice(ctx->device));
    uint32_t h[4] = {0, 0, 0, 0};
    VX_CUDA(ctx, cudaMemcpyAsync(h, ctx->multi_status.ptr, 16, cudaMemcpyDeviceToHost, ctx->stream));
    VX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *timed_out = (int32_t)h[0];
    if (h[0]) {
        VX_CUDA(ctx, cudaMemsetAsync(ctx->multi_status.ptr, 0, 16, ctx->stream));
        return vx_fail(ctx, VX_ERR_CUDA, "vx_wait_flags timed out: a peer never published the frame");
    }
    return VX_OK;
}

} // extern "C"
