// p2p_api.cu - C ABI (include/p2p.h) over the sm_100a kernels: the single translation unit of libp2p_b200.so.
//   p2p_ctx.cuh          contexts, slots (stream + device buffers), error / allocation helpers
//   p2p_api_project.inl  projection path: upload / pack, launches, view lists, replication across contexts
//   p2p_api_jpeg.inl     JPEG encoder host side         p2p_api_jpegdec.inl  JPEG decoder host side
//   p2p_api_png.inl      PNG encoder host side          p2p_api_pngdec.inl   PNG decoder host side
//   p2p_api_files.inl    files flows: the entry points that return encoded files (encode, project and encode)
// and, below, life cycle, options, host helpers, streams / events and the stage-isolated debug exports.
#include "p2p_ctx.cuh"

#include "p2p_api_project.inl"
#include "p2p_api_jpeg.inl"
#include "p2p_api_jpegdec.inl"
#include "p2p_api_png.inl"
#include "p2p_api_pngdec.inl"
#include "p2p_api_files.inl"

// ============================================================================================
extern "C" {

int p2p_abi_version(void) { return P2P_ABI_VERSION; }

int p2p_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char *p2p_status_string(int status) {
    switch (status) {
        case P2P_OK: return "ok";
        case P2P_ERR_INVALID: return "invalid argument";
        case P2P_ERR_CUDA: return "CUDA error";
        case P2P_ERR_NOMEM: return "out of memory";
        case P2P_ERR_STATE: return "bad slot state";
        case P2P_ERR_LIMIT: return "size limit exceeded";
        case P2P_ERR_UNSUPPORTED: return "file outside the supported subset (use cv2.imread)";
        default: return "unknown status";
    }
}

int p2p_create(int device, int n_slots, p2p_ctx **out) {
    if (!out || n_slots <= 0 || n_slots > 64) return P2P_ERR_INVALID;
    *out = nullptr;
    int n = p2p_device_count();
    if (n <= 0 || device < 0 || device >= n) return P2P_ERR_CUDA;  // no CPU fallback
    p2p_ctx *ctx = new (std::nothrow) p2p_ctx;
    if (!ctx) return P2P_ERR_NOMEM;
    ctx->device = device;
    ctx->n_slots = n_slots;
    ctx->slots = new (std::nothrow) Slot[n_slots];
    if (!ctx->slots) {
        delete ctx;
        return P2P_ERR_NOMEM;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        cudaGetLastError();
        delete[] ctx->slots;
        delete ctx;
        return P2P_ERR_CUDA;
    }
    for (int i = 0; i < n_slots; ++i) {
        if (cudaStreamCreateWithFlags(&ctx->slots[i].stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError();
            for (int j = 0; j < i; ++j) cudaStreamDestroy(ctx->slots[j].stream);
            delete[] ctx->slots;
            delete ctx;
            return P2P_ERR_CUDA;
        }
        ctx->slots[i].own_stream = true;
    }
    *out = ctx;
    return P2P_OK;
}

void p2p_destroy(p2p_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < ctx->n_slots; ++i) {
        Slot &s = ctx->slots[i];
        if (s.wait_ev) cudaEventDestroy(s.wait_ev);
        if (s.tex) cudaDestroyTextureObject(s.tex);
        if (s.surf) cudaDestroySurfaceObject(s.surf);
        if (s.arr) cudaFreeArray(s.arr);
        for (int c = 0; c < 3; ++c) {
            if (s.ftex[c]) cudaDestroyTextureObject(s.ftex[c]);
            if (s.fsurf[c]) cudaDestroySurfaceObject(s.fsurf[c]);
            if (s.farr[c]) cudaFreeArray(s.farr[c]);
        }
        cudaFree(s.d_bgr);
        cudaFree(s.d_rgba);
        cudaFree(s.d_out);
        cudaFree(s.d_tab);
        cudaFree(s.j_coef);
        cudaFree(s.j_bits);
        cudaFree(s.j_stream);
        cudaFree(s.j_cnt);
        cudaFree(s.j_out);
        cudaFree(s.j_tot);
        if (s.j_sizes_h) cudaFreeHost(s.j_sizes_h);
        if (s.jd_coef_h) cudaFreeHost(s.jd_coef_h);
        cudaFree(s.jd_coef_d);
        cudaFree(s.jd_planes);
        cudaFree(s.pg_F);
        cudaFree(s.pg_tlen);
        cudaFree(s.pg_blk);
        cudaFree(s.pg_info);
        cudaFree(s.pg_Z);
        cudaFree(s.pg_sums);
        cudaFree(s.jd_stream);
        cudaFree(s.jd_raw);
        cudaFree(s.jd_dcnt);
        cudaFree(s.jd_gate_d);
        cudaFree(s.jd_states);
        cudaFree(s.jd_nblk);
        cudaFree(s.jd_tables);
        cudaFree(s.jd_dc);
        cudaFree(s.jd_tiles);
        cudaFree(s.jd_tot_d);
        cudaFree(s.jd_sub);
        if (s.jd_flags_h) cudaFreeHost(s.jd_flags_h);
        if (s.pd_zs_h) cudaFreeHost(s.pd_zs_h);
        if (s.pd_tab_h) cudaFreeHost(s.pd_tab_h);
        cudaFree(s.pd_zs);
        cudaFree(s.pd_tab);
        cudaFree(s.pd_raw);
        cudaFree(s.pd_ref);
        cudaFree(s.pd_match);
        if (s.own_stream && s.stream) cudaStreamDestroy(s.stream);
        if (s.owned) cudaStreamDestroy(s.owned);
    }
    cudaFree(ctx->d_flush);
    cudaFree(ctx->d_range);
    for (const p2p_ctx::JTab &t : ctx->jtabs) cudaFree(t.d);
    cudaFree(ctx->d_crc_table);
    cudaGetLastError();
    delete[] ctx->slots;
    delete ctx;
}

const char *p2p_last_error(p2p_ctx *ctx) {
    if (!ctx) return "null context";
    return (tl_err_ctx == ctx) ? tl_err.c_str() : "";  // valid until this thread's next failing call
}

int p2p_set_option(p2p_ctx *ctx, int key, int value) {
    if (!ctx) return P2P_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    switch (key) {
        case P2P_OPT_SAMPLER:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "sampler must be 0 or 1");
            ctx->opt_sampler = value;
            return P2P_OK;
        case P2P_OPT_WARP_W:
            if (value != 8 && value != 32) return fail(ctx, P2P_ERR_INVALID, "warp_w must be 8 or 32");
            ctx->opt_warp_w = value;
            return P2P_OK;
        case P2P_OPT_YAWS_PER_THREAD:
            if (value < 1 || value > 4) return fail(ctx, P2P_ERR_INVALID, "yaws per thread must be 1..4");
            ctx->opt_ny = value;
            return P2P_OK;
        case P2P_OPT_IMAGES_PER_LAUNCH:
            if (value != 1 && value != 2 && value != 4) return fail(ctx, P2P_ERR_INVALID, "images per launch must be 1, 2 or 4");
            ctx->opt_nb = value;
            return P2P_OK;
        case P2P_OPT_MIRROR:
            if (value < 0 || value > 2) return fail(ctx, P2P_ERR_INVALID, "mirror must be 0, 1 or 2");
            ctx->opt_mirror = value;
            return P2P_OK;
        case P2P_OPT_SEG_CHUNKS:
            if (value < 1 || value > 64) return fail(ctx, P2P_ERR_INVALID, "seg_chunks must be 1..64");
            ctx->opt_seg_chunks = value;
            return P2P_OK;
        case P2P_OPT_INTERP:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "interp must be 0 (cv2 fixed point) or 1 (exact bilinear)");
            ctx->opt_interp = value;
            return P2P_OK;
        case P2P_OPT_SEAM_WRAP:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "seam_wrap must be 0 or 1");
            ctx->opt_seam_wrap = value;
            return P2P_OK;
        case P2P_OPT_TRIG:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "trig must be 0 (NumPy-exact) or 1 (minimax)");
            ctx->opt_trig = value;
            return P2P_OK;
        case P2P_OPT_PARTIAL_UPLOAD:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "partial_upload must be 0 or 1");
            ctx->opt_partial = value;
            return P2P_OK;
        case P2P_OPT_HOST_WAIT:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "host_wait must be 0 or 1");
            ctx->opt_host_wait.store(value);
            return P2P_OK;
        case P2P_OPT_PNG_FORMATS:
            if (value != 0 && value != 1) return fail(ctx, P2P_ERR_INVALID, "png_formats must be 0 or 1");
            ctx->opt_png_formats.store(value);
            return P2P_OK;
        case P2P_OPT_GPU_HUFFMAN:
            if (value < 0 || value > 3) return fail(ctx, P2P_ERR_INVALID, "gpu_huffman must be 0 ... 3");
            ctx->opt_gpu_huffman = value;
            return P2P_OK;
        case P2P_OPT_POISON:
            if (value < -1 || value > 255) return fail(ctx, P2P_ERR_INVALID, "poison must be -1 (off) or a byte 0 ... 255");
            ctx->opt_poison.store(value);
            return P2P_OK;

        default:
            return fail(ctx, P2P_ERR_INVALID, "unknown option");
    }
}

int p2p_get_option(p2p_ctx *ctx, int key, int *value) {
    if (!ctx || !value) return P2P_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    switch (key) {
        case P2P_OPT_SAMPLER: *value = ctx->opt_sampler; return P2P_OK;
        case P2P_OPT_WARP_W: *value = ctx->opt_warp_w; return P2P_OK;
        case P2P_OPT_YAWS_PER_THREAD: *value = ctx->opt_ny; return P2P_OK;
        case P2P_OPT_COUNT_LAUNCHES: *value = (int)ctx->launches; return P2P_OK;
        case P2P_OPT_IMAGES_PER_LAUNCH: *value = ctx->opt_nb; return P2P_OK;
        case P2P_OPT_MIRROR: *value = ctx->opt_mirror; return P2P_OK;
        case P2P_OPT_SEG_CHUNKS: *value = ctx->opt_seg_chunks; return P2P_OK;
        case P2P_OPT_INTERP: *value = ctx->opt_interp; return P2P_OK;
        case P2P_OPT_SEAM_WRAP: *value = ctx->opt_seam_wrap; return P2P_OK;
        case P2P_OPT_TRIG: *value = ctx->opt_trig; return P2P_OK;
        case P2P_OPT_PARTIAL_UPLOAD: *value = ctx->opt_partial; return P2P_OK;
        case P2P_OPT_GPU_HUFFMAN: *value = ctx->opt_gpu_huffman; return P2P_OK;
        case P2P_OPT_HOST_WAIT: *value = ctx->opt_host_wait.load(); return P2P_OK;
        case P2P_OPT_PNG_FORMATS: *value = ctx->opt_png_formats.load(); return P2P_OK;
        case P2P_OPT_GPU_HUFFMAN_COUNT: *value = (int)ctx->gpu_huffman_used; return P2P_OK;
        case P2P_OPT_PNG_HOST_BLOCKS: *value = (int)ctx->png_host_blocks.load(); return P2P_OK;
        case P2P_OPT_POISON: *value = ctx->opt_poison.load(); return P2P_OK;

        default: return fail(ctx, P2P_ERR_INVALID, "unknown option");
    }
}

// ---- host helpers --------------------------------------------------------------------------
int p2p_pitch_constants(double fov_deg, double pitch_deg, int W, p2p_pitch_consts *out) {
    if (!out || W <= 0) return P2P_ERR_INVALID;
    const double deg = M_PI / 180.0;  // np.radians(x) == x * (pi / 180)
    const double fov = fov_deg * deg, p = pitch_deg * deg;
    out->f = (float)((0.5 * (double)W) / tan(fov / 2.0));
    out->c = (float)cos(p);
    out->s = (float)sin(p);
    return P2P_OK;
}

int p2p_yaw_table(int Wp, double yaw_deg, int32_t *ix, int32_t *fx, int32_t *shift) {
    if (Wp <= 0 || !ix || !fx) return P2P_ERR_INVALID;
    const double two_pi = 2.0 * M_PI;
    const double yaw = yaw_deg * (M_PI / 180.0);  // f64 scalar: the sum below is f64 (NEP 50)
    const float two_pi_f = (float)two_pi;
    bool roll = true;
    for (int u = 0; u < Wp; ++u) {
        // ref :95   phi = (2*pi*u / Wp) in f32: f32(2pi) * f32(u), then / f32(Wp)
        volatile float m = two_pi_f * (float)u;
        const float phi = m / (float)Wp;
        // ref :98   (phi + yaw) % 2pi in f64, Python-style remainder (result takes divisor's sign)
        double r = fmod((double)phi + yaw, two_pi);
        if (r != 0.0) {
            if (r < 0.0) r += two_pi;
        } else {
            r = 0.0;
        }
        // ref :101-105
        double U = (r * (double)Wp) / two_pi;
        if (U < 0.0) U = 0.0;
        if (U > (double)(Wp - 1)) U = (double)(Wp - 1);
        const float Uf = (float)U;
        volatile float sc = Uf * 32.0f;
        const int sx = (int)lrintf(sc);  // cvRound: round half even
        ix[u] = sx >> 5;
        fx[u] = sx & 31;
        if (fx[u] != 0) roll = false;
    }
    if (roll) {
        const int s0 = ix[0];
        for (int u = 0; u < Wp && roll; ++u) roll = (ix[u] == (u + s0) % Wp);
        if (shift) *shift = roll ? s0 : -1;
    } else if (shift) {
        *shift = -1;
    }
    return P2P_OK;
}

int p2p_host_alloc(void **ptr, size_t bytes) {
    if (!ptr || bytes == 0) return P2P_ERR_INVALID;
    cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *ptr = nullptr;
        return P2P_ERR_NOMEM;
    }
    return P2P_OK;
}

int p2p_host_free(void *ptr) {
    if (!ptr) return P2P_OK;
    if (cudaFreeHost(ptr) != cudaSuccess) {
        cudaGetLastError();
        return P2P_ERR_CUDA;
    }
    return P2P_OK;
}

int p2p_host_register(void *ptr, size_t bytes) {
    if (!ptr || bytes == 0) return P2P_ERR_INVALID;
    if (cudaHostRegister(ptr, bytes, cudaHostRegisterPortable) != cudaSuccess) {
        cudaGetLastError();
        return P2P_ERR_CUDA;
    }
    return P2P_OK;
}

int p2p_host_unregister(void *ptr) {
    if (!ptr) return P2P_ERR_INVALID;
    if (cudaHostUnregister(ptr) != cudaSuccess) {
        cudaGetLastError();
        return P2P_ERR_CUDA;
    }
    return P2P_OK;
}

int p2p_sync(p2p_ctx *ctx, int slot) {
    if (!ctx) return P2P_ERR_INVALID;
    // the streams are read under the lock, the wait itself happens outside it: a thread waiting for its slot must
    // not keep the other threads (other slots) from enqueueing
    std::vector<cudaStream_t> streams;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (slot >= 0 && !slot_ok(ctx, slot)) return fail(ctx, P2P_ERR_INVALID, "bad slot");
        for (int i = 0; i < ctx->n_slots; ++i)
            if (slot < 0 || i == slot) streams.push_back(ctx->slots[i].stream);
    }
    cudaError_t e = cudaSetDevice(ctx->device);
    for (size_t i = 0; i < streams.size() && e == cudaSuccess; ++i) e = cudaStreamSynchronize(streams[i]);
    if (e != cudaSuccess) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        cudaGetLastError();
        return fail(ctx, P2P_ERR_CUDA, "cudaStreamSynchronize", e);
    }
    return P2P_OK;
}

int p2p_set_stream(p2p_ctx *ctx, int slot, void *cuda_stream) {
    if (!slot_ok(ctx, slot)) return fail(ctx, P2P_ERR_INVALID, "bad slot");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    CK(wait_slot(ctx, s));
    // the slot's own stream is kept (another slot may have borrowed it through p2p_get_stream)
    // and released by p2p_destroy
    if (s.own_stream) s.owned = s.stream;
    s.stream = static_cast<cudaStream_t>(cuda_stream);
    s.own_stream = false;
    return P2P_OK;
}

int p2p_get_stream(p2p_ctx *ctx, int slot, void **cuda_stream) {
    if (!slot_ok(ctx, slot) || !cuda_stream) return fail(ctx, P2P_ERR_INVALID, "bad slot or null pointer");
    std::lock_guard<std::mutex> lk(ctx->mu);
    *cuda_stream = ctx->slots[slot].stream;
    return P2P_OK;
}

// ---- timing --------------------------------------------------------------------------------
int p2p_event_create(p2p_ctx *ctx, void **event) {
    if (!ctx || !event) return P2P_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    *event = e;
    return P2P_OK;
}

int p2p_event_destroy(p2p_ctx *ctx, void *event) {
    if (!ctx || !event) return P2P_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaEventDestroy(static_cast<cudaEvent_t>(event)));
    return P2P_OK;
}

int p2p_event_record(p2p_ctx *ctx, void *event, int slot) {
    if (!slot_ok(ctx, slot) || !event) return fail(ctx, P2P_ERR_INVALID, "bad slot or event");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(static_cast<cudaEvent_t>(event), ctx->slots[slot].stream));
    return P2P_OK;
}

int p2p_event_wait(p2p_ctx *ctx, void *event, int slot) {
    if (!slot_ok(ctx, slot) || !event) return fail(ctx, P2P_ERR_INVALID, "bad slot or null event");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamWaitEvent(ctx->slots[slot].stream, static_cast<cudaEvent_t>(event), 0));
    return P2P_OK;
}

int p2p_event_elapsed_ms(p2p_ctx *ctx, void *start, void *stop, float *ms) {
    if (!ctx || !start || !stop || !ms) return P2P_ERR_INVALID;
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventSynchronize(static_cast<cudaEvent_t>(stop)));
    CK(cudaEventElapsedTime(ms, static_cast<cudaEvent_t>(start), static_cast<cudaEvent_t>(stop)));
    return P2P_OK;
}

int p2p_flush_l2(p2p_ctx *ctx, int slot, size_t bytes) {
    if (!slot_ok(ctx, slot) || bytes == 0) return fail(ctx, P2P_ERR_INVALID, "bad slot or size");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    bytes = (bytes + 15) & ~(size_t)15;
    int rc = ensure(ctx, &ctx->d_flush, &ctx->flush_cap, bytes);
    if (rc) return rc;
    fill_kernel<<<148 * 8, 256, 0, ctx->slots[slot].stream>>>(ctx->d_flush, bytes / 16, (uint32_t)ctx->launches);
    ctx->launches++;
    CK(cudaGetLastError());
    return P2P_OK;
}

// ---- debug exports -------------------------------------------------------------------------
int p2p_selftest(p2p_ctx *ctx, const p2p_pitch_consts *pitch, int W, int H, int exhaustive_div,
                 unsigned long long *ray_mismatches, unsigned long long *div_mismatches) {
    if (!ctx || !pitch || W <= 0 || H <= 0 || !ray_mismatches || !div_mismatches)
        return fail(ctx, P2P_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CK(cudaSetDevice(ctx->device));
    unsigned long long *d = nullptr;
    CK(cudaMalloc(&d, 2 * sizeof(unsigned long long)));
    cudaStream_t st = ctx->slots[0].stream;
    cudaError_t e = cudaMemsetAsync(d, 0, 2 * sizeof(unsigned long long), st);
    if (e == cudaSuccess) {
        PitchC k{pitch->f, pitch->c, pitch->s};
        dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
        selftest_ray_kernel<<<grid, block, 0, st>>>(k, W, H, (float)(W / 2.0), (float)(H / 2.0), d);
        ctx->launches++;
        if (exhaustive_div) {
            selftest_constdiv_kernel<<<148 * 16, 256, 0, st>>>(d);
            ctx->launches++;
        }
        e = cudaGetLastError();
    }
    unsigned long long h[2] = {0, 0};
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, P2P_ERR_CUDA, "p2p_selftest", e);
    *ray_mismatches = h[0];
    *div_mismatches = h[1];
    return P2P_OK;
}

int p2p_coords(p2p_ctx *ctx, const p2p_pitch_consts *pitch, int W, int H, int Wp, int Hp,
               float *U_host, float *V_host) {
    if (!ctx || !pitch || !U_host || !V_host || W <= 0 || H <= 0) return fail(ctx, P2P_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc = check_dims(ctx, Wp, Hp);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)W * H;
    float *d = nullptr;
    CK(cudaMalloc(&d, n * 2 * sizeof(float)));
    PitchC k{pitch->f, pitch->c, pitch->s};
    dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    cudaStream_t st = ctx->slots[0].stream;
    coords_kernel<<<grid, block, 0, st>>>(k, W, H, (float)(W / 2.0), (float)(H / 2.0), (float)Wp, (float)Hp,
                                          (float)(Wp - 1), (float)(Hp - 1), d, d + n, ctx->opt_trig == 0);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(U_host, d, n * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(V_host, d + n, n * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, P2P_ERR_CUDA, "p2p_coords", e);
    return P2P_OK;
}

int p2p_sample_with_maps(p2p_ctx *ctx, int slot, int yaw_shift, const float *U_host, const float *V_host,
                         int W, int H, uint8_t *out_host) {
    if (!slot_ok(ctx, slot) || !U_host || !V_host || !out_host || W <= 0 || H <= 0)
        return fail(ctx, P2P_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    Slot &s = ctx->slots[slot];
    if (!s.valid) return fail(ctx, P2P_ERR_STATE, "slot holds no panorama");
    if (yaw_shift < 0 || yaw_shift >= s.Wp) return fail(ctx, P2P_ERR_INVALID, "yaw_shift outside [0, Wp)");
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)W * H;
    float *d = nullptr;
    uint8_t *d_o = nullptr;
    CK(cudaMalloc(&d, n * 2 * sizeof(float)));
    cudaError_t e = cudaMalloc(&d_o, n * 3);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d, U_host, n * sizeof(float), cudaMemcpyHostToDevice, s.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + n, V_host, n * sizeof(float), cudaMemcpyHostToDevice, s.stream);
    if (e == cudaSuccess) {
        dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
        sample_maps_kernel<<<grid, block, 0, s.stream>>>(s.d_rgba, s.pitch_tex, s.Wp, s.Hp, yaw_shift, d, d + n, W, H, d_o,
                                                        ctx->opt_interp, ctx->opt_interp == 1 && ctx->opt_seam_wrap);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_host, d_o, n * 3, cudaMemcpyDeviceToHost, s.stream);
    if (e == cudaSuccess) e = wait_slot(ctx, s);
    cudaFree(d);
    cudaFree(d_o);
    if (e != cudaSuccess) return fail(ctx, P2P_ERR_CUDA, "p2p_sample_with_maps", e);
    return P2P_OK;
}

int p2p_download_pano(p2p_ctx *ctx, int slot, uint8_t *bgr_host, size_t row_stride) {
    if (!slot_ok(ctx, slot) || !bgr_host) return fail(ctx, P2P_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    Slot &s = ctx->slots[slot];
    if (!s.valid) return fail(ctx, P2P_ERR_STATE, "slot holds no panorama");
    if (slot_is_partial(s)) return fail(ctx, P2P_ERR_STATE, "slot holds a partial panorama (p2p_process_image)");
    if (row_stride < (size_t)s.Wp * 3) return fail(ctx, P2P_ERR_INVALID, "row_stride smaller than Wp * 3");
    CK(cudaSetDevice(ctx->device));
    uint8_t *d = nullptr;
    const size_t dstride = (size_t)s.Wp * 3;
    CK(cudaMalloc(&d, dstride * s.Hp));
    dim3 block(256), grid((s.Wp + 255) / 256, s.Hp);
    unpack_kernel<<<grid, block, 0, s.stream>>>(s.d_rgba, s.pitch_tex, s.Wp, s.Hp, d, dstride);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = cudaMemcpy2DAsync(bgr_host, row_stride, d, dstride, dstride, s.Hp, cudaMemcpyDeviceToHost, s.stream);
    if (e == cudaSuccess) e = wait_slot(ctx, s);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, P2P_ERR_CUDA, "p2p_download_pano", e);
    return P2P_OK;
}

int p2p_debug_poison(p2p_ctx *ctx, int slot, int byte) {
    if (!slot_ok(ctx, slot) || byte < 0 || byte > 255) return fail(ctx, P2P_ERR_INVALID, "bad slot or byte");
    std::lock_guard<std::mutex> lk(ctx->mu);
    Slot &s = ctx->slots[slot];
    if (s.jd_run.pending) return fail(ctx, P2P_ERR_STATE, "a JPEG decode's Huffman verdict is still pending on the slot");
    CK(cudaSetDevice(ctx->device));
    CK(wait_slot(ctx, s));
    const cudaStream_t st = s.stream;
    const struct { void *p; size_t n; } scratch[] = {
        {s.d_bgr, s.bgr_cap}, {s.d_out, s.out_cap}, {s.d_tab, s.tab_cap},
        {s.j_coef, s.j_coef_cap}, {s.j_bits, s.j_bits_cap}, {s.j_stream, s.j_stream_cap}, {s.j_cnt, s.j_cnt_cap},
        {s.j_out, s.j_out_cap}, {s.j_tot, s.j_tot_cap},
        {s.pg_F, s.pg_F_cap}, {s.pg_tlen, s.pg_tlen_cap}, {s.pg_blk, s.pg_blk_cap}, {s.pg_info, s.pg_info_cap},
        {s.pg_Z, s.pg_Z_cap}, {s.pg_sums, s.pg_sums_cap},
        {s.jd_coef_d, s.jd_coef_d_cap}, {s.jd_planes, s.jd_planes_cap}, {s.jd_stream, s.jd_stream_cap},
        {s.jd_states, s.jd_states_cap}, {s.jd_nblk, s.jd_nblk_cap}, {s.jd_tables, sizeof(p2pjdec::DevTables)},
        {s.jd_dc, s.jd_dc_cap}, {s.jd_tiles, s.jd_tiles_cap}, {s.jd_tot_d, 4 * sizeof(unsigned long long)},
        {s.jd_raw, s.jd_raw_cap}, {s.jd_dcnt, s.jd_dcnt_cap}, {s.jd_gate_d, 8 * sizeof(int)}, {s.jd_sub, s.jd_sub_cap},
        {s.pd_zs, s.pd_zs_cap}, {s.pd_tab, s.pd_tab_cap}, {s.pd_raw, s.pd_raw_cap}, {s.pd_ref, s.pd_ref_cap},
        {s.pd_match, s.pd_match_cap},
    };
    for (const auto &b : scratch)
        if (b.p) CK(cudaMemsetAsync(b.p, byte, b.n, st));
    // the panorama: packed rows row0 .. row1 hold it (columns 0 .. Wp: the wrap column included)
    const bool held = s.valid && s.d_rgba;
    if (s.d_rgba) {
        uint8_t *base = reinterpret_cast<uint8_t *>(s.d_rgba);
        const size_t row = (size_t)s.pitch_tex * 4;
        const size_t a = held ? row * s.row0 : 0, b = held ? row * (s.row1 + 1) : 0;
        if (a) CK(cudaMemsetAsync(base, byte, a, st));
        if (s.rgba_cap > b) CK(cudaMemsetAsync(base + b, byte, s.rgba_cap - b, st));
        if (held && s.pitch_tex > s.Wp + 1)
            CK(cudaMemset2DAsync(base + a + (size_t)(s.Wp + 1) * 4, row, byte, (size_t)(s.pitch_tex - s.Wp - 1) * 4,
                                 (size_t)(s.row1 - s.row0 + 1), st));
    }
    // the gather array and the folded planes hold rows row0 .. min(row1, Hp - 1) while they are current
    const int k1 = (s.row1 < s.Hp - 1) ? s.row1 : s.Hp - 1;
    if (s.arr) {
        const bool keep = held && s.tex_current;
        int rc = poison_array(ctx, s.surf, s.arrW, s.arrH, keep ? s.row0 : 1, keep ? k1 : 0, byte, st);
        if (rc) return rc;
    }
    for (int c = 0; c < 3; ++c) {
        if (!s.farr[c]) continue;
        const bool keep = held && s.fold_current;
        int rc = poison_array(ctx, s.fsurf[c], s.farrW, s.farrH, keep ? s.row0 : 1, keep ? k1 : 0, byte, st);
        if (rc) return rc;
    }
    CK(wait_slot(ctx, s));
    // pinned and mapped host buffers (no kernel of the slot runs any more)
    if (s.jd_coef_h) memset(s.jd_coef_h, byte, s.jd_coef_h_cap);
    if (s.pd_zs_h) memset(s.pd_zs_h, byte, s.pd_zs_h_cap);
    if (s.pd_tab_h) memset(s.pd_tab_h, byte, s.pd_tab_h_cap);
    if (s.j_sizes_h) memset(s.j_sizes_h, byte, (size_t)s.j_sizes_n * sizeof(unsigned long long));
    if (s.jd_flags_h) memset(s.jd_flags_h, byte, sizeof(*s.jd_flags_h));
    return P2P_OK;
}

}  // extern "C"
