// host_objects.cuh -- part of the C-ABI translation unit (included by lwb_api.cu, not compiled on its own):
// the opaque objects behind the handles (ctx, setup, stream, plan), error / buffer helpers and the
// window geometry of audio.rs:1056-1073.
#pragma once

// ---------------------------------------------------------------------------------------------
// objects
// ---------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

// pinned staging for one batch's descriptors; `ev` marks the end of the copy that reads it
struct Staging {
    void *h = nullptr;
    size_t cap = 0;
    cudaEvent_t ev = nullptr;
    bool pending = false;
};

// CachedBlocksizeDerived (header_cached.rs:27-31) on the device, shared by all setups of a context with the same tables
struct CachedTables {
    DevTables dt;                  // device pointers; dt.pack = the fused kernels' twiddle pack (bs 11: k_long, bs 8: k_short)
    std::vector<float> a, b, c, w; // host copies: the cache key
    std::vector<uint32_t> br;
    std::vector<void *> allocs;
};

struct lwb_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t ev_in[64] = {}, ev_done[65] = {};      // per chunk of a host-memory batch; [64] orders the copy streams
    // fused path: descriptor arrays are double buffered and uploaded on the copy stream so that the
    // upload of step k+1 overlaps kernel k; tickets come from a pool zeroed once per wrap
    DevBuf runs_buf[2];
    cudaEvent_t ev_desc[2] = {}, ev_kdone[2] = {};
    int runs_par = 0;
    uint32_t ticket_next = 0;
    uint64_t epoch = 0;            // batch counter: lwb_stream::busy_epoch == epoch <=> the stream already sits in this batch
    uint64_t state_gen = 1;        // bumped whenever any stream's (has, len) changes: plans key on it
    std::string err;
    uint64_t launches = 0;
    uint64_t long_launches = 0;    // of which k_long / k_long_s
    std::deque<CachedTables> tables;       // (deque: setups hold copies of dt, growth never moves an entry)
    // grow-only device arenas
    DevBuf coeffs, dense, pcm, spec, segtab, vqoff, vqrec, magic, x, desc, kinds, ys, chains, ticket, cdesc, cbytes;
    Staging stage[3];              // ring: a batch's descriptors are written while the previous copies may still run
    int stage_next = 0;
    // pinned staging for descriptors (four-kernel path)
    void *h_desc = nullptr;
    size_t h_desc_cap = 0;
    size_t x_cap_elems = (size_t)64 << 20;     // IMDCT scratch per round of the generic path (256 MiB)
};

struct lwb_setup {
    lwb_ctx *ctx = nullptr;
    DevSetup host;                 // device pointers inside
    DevSetup *d_setup = nullptr;
    std::vector<void *> allocs;
    uint8_t channels = 0, bs0 = 0, bs1 = 0;
    uint32_t n_modes = 0;
    uint32_t n_mappings = 0;
    std::vector<DevMapping> mappings;   // host copy (validation)
};

struct MixRound { size_t r0, nr, s0, ns, c0, nc, x0, nx, g0, ng, flat, nm; };   // LongRun / ShortRun / ChainDesc / RowCopy / burst-group ranges of one
                                                                            // round; flat: the one-pass round (static deal, k_long_s);
                                                                            // nm: groups of k_mid (path_mid.cuh, from the buffer's start)
struct RowCopy { const float *src; float *dst; uint32_t n4, pad; };  // n4 float4s, copied in front of the round's kernels
struct MixLaunch {
    char *db; size_t off_sr, off_cd, off_by, off_rc, off_sg;
    const float *pack, *spack, *w_short, *mpack; int ls, mid_kb; bool i16, residue; int out_format; unsigned warps; size_t smem; int n1max, wpc, np;
    const float *coeffs, *dense; const uint8_t *kinds; const uint32_t *ys; void *pcm;
};

struct lwb_plan {
    lwb_ctx *ctx = nullptr;
    lwb_chain *chains = nullptr;
    size_t n_chains = 0;
    lwb_batch_io io;
    // captured fused-path launch (valid while ctx->state_gen == gen)
    bool captured = false;
    uint64_t gen = 0;
    DevBuf runs;
    uint32_t n_groups = 0;
    const float *pack = nullptr;
    bool i16 = false;
    int step = 1;                  // k_long's PCM step: 1 planar, the channel count interleaved
    // residue entry: the front-stage descriptors (one DevPacket per packet).  They depend only on the captured
    // chain / mode arrays, never on stream state, so they stay valid for the plan's lifetime.
    bool pro_captured = false, pro_fast = false;
    DevBuf pro;
    size_t n_pro = 0, pro_smem_old = 0;
    unsigned pro_C = 0;
    uint64_t pro_c_lo = 0, pro_c_hi = 0, pro_r_lo = 0, pro_r_hi = 0;
    // captured mixed-path launch sequence (valid while ctx->state_gen == gen)
    bool mixed_captured = false;
    DevBuf mix;
    MixLaunch mix_launch;
    std::vector<MixRound> mix_rounds;
    // ... residue entry: its front-stage descriptors sit in `mix` too
    bool mix_pro = false, mix_pro_fast = false, mix_pro_dense = false;
    const DevPacket *mix_pro_pk = nullptr;
    size_t mix_pro_n = 0, mix_pro_smem_old = 0;
    unsigned mix_pro_C = 0;
    int mix_pro_n2max = 0;
    uint64_t mix_pro_c_lo = 0, mix_pro_r_lo = 0, mix_pro_r_hi = 0;
};

struct lwb_stream {
    lwb_ctx *ctx = nullptr;
    const lwb_setup *setup = nullptr;
    float *d_state = nullptr;      // [channels][n1/2]
    bool has = false;              // PreviousWindowRight.data.is_some()
    uint32_t plen = 0;             // per-channel length of the saved right half
    uint64_t busy_epoch = 0;       // guards against one stream appearing twice in a batch
};

static inline void set_stream_state(lwb_stream *s, bool has, uint32_t plen)
{
    if (s->has != has || s->plen != plen) {
        s->has = has;
        s->plen = plen;
        s->ctx->state_gen++;
    }
}

static int fail(lwb_ctx *ctx, int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (ctx) {
        ctx->err = what;
        if (e != cudaSuccess) {
            ctx->err += ": ";
            ctx->err += cudaGetErrorString(e);
        }
    }
    return code;
}

#define CU(ctx, call)                                                        \
    do {                                                                     \
        cudaError_t e__ = (call);                                            \
        if (e__ != cudaSuccess) return fail((ctx), LWB_ERR_CUDA, #call, e__); \
    } while (0)

static int ensure(lwb_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return LWB_OK;
    if (b.p) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        CU(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 4096;
    CU(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    ctx->state_gen++;              // captured plans may hold pointers into the arena that just moved
    return LWB_OK;
}

static int ensure_pinned(lwb_ctx *ctx, size_t bytes)
{
    if (bytes <= ctx->h_desc_cap) return LWB_OK;
    if (ctx->h_desc) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFreeHost(ctx->h_desc);
        ctx->h_desc = nullptr;
        ctx->h_desc_cap = 0;
    }
    size_t want = bytes * 2 + 4096;
    CU(ctx, cudaHostAlloc(&ctx->h_desc, want, cudaHostAllocDefault));
    ctx->h_desc_cap = want;
    return LWB_OK;
}

// ---------------------------------------------------------------------------------------------
// window geometry, audio.rs:1056-1073 (and its twin :889-908)
// ---------------------------------------------------------------------------------------------
struct Geom {
    uint32_t n, ls, le, rs, re;
    uint8_t blockflag, slope_sel, mapping;
};

static int geometry(const lwb_setup *su, uint8_t mode, int prev_flag, int next_flag, Geom *g)
{
    if (mode >= su->n_modes) return LWB_ERR_BAD_FORMAT;          // audio.rs:926-930
    const bool lng = su->host.mode_blockflag[mode] != 0;
    const uint32_t n = 1u << (lng ? su->bs1 : su->bs0);
    const uint32_t n0 = 1u << su->bs0;
    const bool prev = lng ? (prev_flag != 0) : true;             // short blocks: map_or(true, ..)
    const bool next = lng ? (next_flag != 0) : true;
    g->n = n;
    g->blockflag = lng;
    g->mapping = su->host.mode_mapping[mode];
    if (prev) { g->ls = 0; g->le = n >> 1; g->slope_sel = lng; }
    else { g->ls = (n - n0) >> 2; g->le = (n + n0) >> 2; g->slope_sel = 0; }
    if (next) { g->rs = n >> 1; g->re = n; }
    else { g->rs = (n * 3 - n0) >> 2; g->re = (n * 3 + n0) >> 2; }
    return LWB_OK;
}

