// path_chain.cuh -- part of the C-ABI translation unit (included by lwb_api.cu, not compiled on its own):
// the chain-kernel path (kernel_chain.cuh) and the launch sequence shared with the mixed path.
#pragma once

// ---------------------------------------------------------------------------------------------
// Chain kernel path (kernel_chain.cuh): everything the fused long-block kernel does not take,
// as long as channels <= 8 and the per-channel buffers fit in shared memory.
// ---------------------------------------------------------------------------------------------
// Shared memory of the chain kernel: per channel `np` blocks of U | V plus the previous right half, and the
// floor posts of up to 8 channels.  np (blocks a channel group transforms together) is 4 where that fits.
static size_t chain_smem(unsigned maxc, int n1max, int np)
{
    return (size_t)maxc * ((size_t)np * n1max + n1max / 2) * 4 + 8 * (LWB_MAX_POSTS + 1) * 2 * 2 + 64;
}
static int chain_np(unsigned maxc, int n1max, int wpc, bool residue)
{
    if (residue || wpc != 1 || getenv("LWB_CHAIN_NP1")) return 1;
    int np = 4;
    while (np > 1 && chain_smem(maxc, n1max, np) > 64 * 1024) np >>= 1;
    return np;
}

template <int ENTRY>
static int launch_chain(lwb_ctx *ctx, int fmt, unsigned n_chains, unsigned warps, size_t smem, const ChainDesc *d,
                        const uint8_t *bytes, const float *coeffs, const float *dense, const uint8_t *kinds,
                        const uint32_t *ys, void *pcm, int n1max, int wpc, int np)
{
#define LWB_CHAIN_CASE(F)                                                                                    \
    case F:                                                                                                  \
        if (wpc == 1) {                                                                                      \
            cudaFuncSetAttribute(k_chain<F, ENTRY, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            return launch(ctx, k_chain<F, ENTRY, false>, dim3(n_chains), dim3(warps * 32), smem, d, bytes, coeffs, dense, \
                          kinds, ys, pcm, n1max, wpc, np);                                                    \
        }                                                                                                    \
        cudaFuncSetAttribute(k_chain<F, ENTRY, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        return launch(ctx, k_chain<F, ENTRY, true>, dim3(n_chains), dim3(warps * 32), smem, d, bytes, coeffs, dense, kinds, \
                      ys, pcm, n1max, wpc, 1);
    switch (fmt) {
        LWB_CHAIN_CASE(LWB_OUT_F32_PLANAR)
        LWB_CHAIN_CASE(LWB_OUT_I16_PLANAR)
        LWB_CHAIN_CASE(LWB_OUT_F32_INTERLEAVED)
        LWB_CHAIN_CASE(LWB_OUT_I16_INTERLEAVED)
    }
#undef LWB_CHAIN_CASE
    return LWB_ERR_INVALID;
}

// one launch of the fused kernel and one of the chain kernel per round, in stream order
// One block per row: the stream state the first segment of a chain starts from, moved out of the way of the segment of
// the same chain that ends the batch -- in the one-pass schedule (path_mixed.cuh) that one may store the new state before
// the first one has read the old.
__global__ void k_row_copy(const RowCopy *__restrict__ rc)
{
    const RowCopy c = rc[blockIdx.x];
    for (uint32_t i = threadIdx.x; i < c.n4; i += blockDim.x)
        reinterpret_cast<float4 *>(c.dst)[i] = reinterpret_cast<const float4 *>(c.src)[i];
}

static int mixed_launch_rounds(lwb_ctx *ctx, const MixLaunch &ml, const std::vector<MixRound> &rounds)
{
    constexpr uint32_t kTicketPool = 1024;
    cudaStream_t sm = ctx->stream;
    int rc = LWB_OK;
    for (const MixRound &rd : rounds) {
        if (rd.nm) {             // uniform 1024-point batches (path_mid.cuh)
            if (mid_launch(sm, (const LongRun *)ml.db, (uint32_t)rd.nm, ml.mpack, ctx->sm_count, ml.i16, ml.mid_kb))
                return fail(ctx, LWB_ERR_CUDA, "mid kernel launch", cudaGetLastError());
            ctx->launches++;
        }
        if (rd.nx) {
            k_row_copy<<<(unsigned)rd.nx, 64, 0, sm>>>((const RowCopy *)(ml.db + ml.off_rc) + rd.x0);
            if (cudaGetLastError() != cudaSuccess) return fail(ctx, LWB_ERR_CUDA, "row copy launch", cudaGetLastError());
            ctx->launches++;
        }
        if (rd.nr) {
            if (ctx->ticket_next % kTicketPool == 0)
                CU(ctx, cudaMemsetAsync(ctx->ticket.p, 0, kTicketPool * sizeof(unsigned int), sm));
            unsigned int *ticket = (unsigned int *)ctx->ticket.p + (ctx->ticket_next++ % kTicketPool);
            if (kLongNB != 1) return fail(ctx, LWB_ERR_INVALID, "mixed path needs one run per warp");
            // one pass over many short runs: the static deal with its deeper lookahead (k_long_s); rounds: tickets
            if (rd.flat ? long_launch_static(sm, (const LongRun *)ml.db + rd.r0, (uint32_t)rd.nr, ml.pack, ctx->sm_count, ml.i16, ml.w_short, ml.ls)
                        : long_launch(sm, (const LongRun *)ml.db + rd.r0, (uint32_t)rd.nr, ml.pack, ticket, ctx->sm_count, ml.i16, ml.w_short, ml.ls))
                return fail(ctx, LWB_ERR_CUDA, "long kernel launch", cudaGetLastError());
            ctx->launches++;
            ctx->long_launches++;
        }
        if (rd.ns) {
            if (short_launch(sm, (const ShortRun *)(ml.db + ml.off_sr) + rd.s0, (uint32_t)rd.ns, ml.spack, ctx->sm_count, ml.i16))
                return fail(ctx, LWB_ERR_CUDA, "short kernel launch", cudaGetLastError());
            ctx->launches++;
        }
        if (rd.ng) {             // bursts: eight short runs of equal length per warp (k_short_g)
            if (short_launch_groups(sm, (const ShortRun *)(ml.db + ml.off_sg) + rd.g0 * kShortOct, (uint32_t)rd.ng, ml.spack, ctx->sm_count, ml.i16))
                return fail(ctx, LWB_ERR_CUDA, "short burst kernel launch", cudaGetLastError());
            ctx->launches++;
        }
        if (rd.nc) {
            const ChainDesc *dcd = (const ChainDesc *)(ml.db + ml.off_cd) + rd.c0;
            const uint8_t *dby = (const uint8_t *)(ml.db + ml.off_by);
            if (ml.residue)
                rc = launch_chain<LWB_ENTRY_RESIDUE>(ctx, ml.out_format, (unsigned)rd.nc, ml.warps, ml.smem, dcd, dby, ml.coeffs, ml.dense,
                                                     ml.kinds, ml.ys, ml.pcm, ml.n1max, ml.wpc, ml.np);
            else
                rc = launch_chain<LWB_ENTRY_SPECTRUM>(ctx, ml.out_format, (unsigned)rd.nc, ml.warps, ml.smem, dcd, dby, ml.coeffs, ml.dense,
                                                      ml.kinds, ml.ys, ml.pcm, ml.n1max, ml.wpc, ml.np);
            if (rc) return rc;
        }
    }
    return LWB_OK;
}

static int try_chain(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io, uint64_t epoch,
                     bool *handled, lwb_plan *plan = nullptr)
{
    *handled = false;
    const uint64_t gen_at_entry = ctx->state_gen;
    if (plan) plan->mixed_captured = false;
    if (const char *e = getenv("LWB_FORCE_GENERIC"))
        if (std::strcmp(e, "1") == 0) return LWB_OK;          // "1": the four-kernel path; "2": no fused kernel only
    if (io->entry == LWB_ENTRY_VQ) return LWB_OK;            // (its residue stage runs inside the kernel, on dense vectors)
    const bool residue = io->entry == LWB_ENTRY_RESIDUE;
    const bool planar = is_planar(io->out_format);
    const size_t esz = elem_size(io->out_format);
    unsigned maxc = 1;
    int n1max = 64;
    size_t total_packets = 0;
    for (size_t i = 0; i < n_chains; i++) {
        const lwb_chain *c = &chains[i];
        if (!c->stream || c->stream->ctx != ctx || (c->n_packets && !c->mode_numbers)) return LWB_OK;   // generic path reports it
        const lwb_setup *su = c->stream->setup;
        if (su->channels > 8) return LWB_OK;
        maxc = std::max<unsigned>(maxc, su->channels);
        n1max = std::max(n1max, 1 << su->bs1);
        total_packets += c->n_packets;
    }
    if (chain_smem(maxc, n1max, 1) > 200 * 1024) return LWB_OK;
    // warps per channel: one per 1024 samples of the largest block, at most 32 warps per CTA
    int wpc = std::max(1, std::min(8, n1max / 1024));
    while (wpc > 1 && (unsigned)wpc * maxc > 32) wpc >>= 1;
    const int np = chain_np(maxc, n1max, wpc, residue);
    const size_t smem = chain_smem(maxc, n1max, np);
    if (residue && !io->floor_kind) return fail(ctx, LWB_ERR_INVALID, "residue entry needs floor_kind");
    *handled = true;

    // light walk of every chain: geometry, OLA guard, output size (audio.rs:1056-1073, 1083-1154)
    int rc;
    Staging *st;
    const size_t desc_bytes = n_chains * sizeof(ChainDesc), byte_bytes = total_packets * 3 + 16;
    if ((rc = acquire_staging(ctx, desc_bytes + byte_bytes, &st))) return rc;
    ChainDesc *hd = (ChainDesc *)st->h;
    uint8_t *hb = (uint8_t *)st->h + desc_bytes;
    uint64_t c_lo = ~0ull, c_hi = 0, o_lo = ~0ull, o_hi = 0, r_lo = ~0ull, r_hi = 0;
    int uniform_c = -1;
    bool need_dense = false;
    size_t boff = 0, n_launch = 0;
    struct End { lwb_stream *s; bool has; uint32_t plen; bool touched; };
    std::vector<End> ends(n_chains);
    for (size_t i = 0; i < n_chains; i++) {
        lwb_chain *c = &chains[i];
        lwb_stream *s = c->stream;
        const lwb_setup *su = s->setup;
        if (s->busy_epoch == epoch) return fail(ctx, LWB_ERR_INVALID, "a stream appears in two chains of one batch");
        s->busy_epoch = epoch;
        const unsigned C = su->channels;
        if (residue) {
            if (uniform_c < 0) uniform_c = (int)C;
            if (uniform_c != (int)C) return fail(ctx, LWB_ERR_INVALID, "residue batches need one channel count");
        }
        bool has = s->has, clear_after = false;
        uint32_t plen = s->plen;
        uint64_t coeff = c->coeff_offset, pos = 0;
        uint32_t done = 0;
        c->status = LWB_OK;
        for (uint32_t k = 0; k < c->n_packets; k++) {
            Geom g;
            int grc = geometry(su, c->mode_numbers[k], c->prev_window_flags ? c->prev_window_flags[k] : 1,
                               c->next_window_flags ? c->next_window_flags[k] : 1, &g);
            if (grc) { c->status = grc; break; }
            if (has) {
                const uint32_t slope_len = 1u << ((g.slope_sel ? su->bs1 : su->bs0) - 1);
                if (slope_len < plen) { c->status = LWB_ERR_BAD_FORMAT; clear_after = true; break; }   // audio.rs:1107-1111
                if (g.ls + plen > g.n) { c->status = LWB_ERR_MISMATCH; break; }
                pos += g.rs - g.ls;
            }
            hb[boff + 3 * k] = c->mode_numbers[k];
            hb[boff + 3 * k + 1] = c->prev_window_flags ? c->prev_window_flags[k] : 1;
            hb[boff + 3 * k + 2] = c->next_window_flags ? c->next_window_flags[k] : 1;
            coeff += (uint64_t)C * (g.n >> 1);
            has = true;
            plen = g.re - g.rs;
            done++;
        }
        c->packets_done = done;
        c->n_samples = (uint32_t)pos;
        ends[i] = End{s, clear_after ? false : has, clear_after ? 0u : plen, done > 0 || clear_after};
        if (!done) continue;
        if (planar && c->out_stride < pos) return fail(ctx, LWB_ERR_BUFFER, "chain: out_stride smaller than the samples produced");
        ChainDesc &d = hd[n_launch++];
        std::memset(&d, 0, sizeof(d));
        d.setup = su->d_setup;
        d.state = s->d_state;
        d.coeff_off = c->coeff_offset;
        d.out_off = c->out_offset;
        d.out_stride = c->out_stride;
        d.pkt_index = c->packet_index;
        d.n_packets = done;
        d.byte_off = (uint32_t)boff;
        d.state_stride = (uint32_t)state_stride(su);
        d.plen0 = (uint16_t)s->plen;
        d.has0 = s->has;
        d.channels = (uint8_t)C;
        boff += (size_t)done * 3;
        c_lo = std::min(c_lo, c->coeff_offset);
        c_hi = std::max(c_hi, coeff);
        const uint64_t ext = planar ? (uint64_t)(C - 1) * c->out_stride + pos : pos * C;
        o_lo = std::min(o_lo, c->out_offset);
        o_hi = std::max(o_hi, c->out_offset + ext);
        if (residue) {
            r_lo = std::min(r_lo, c->packet_index);
            r_hi = std::max<uint64_t>(r_hi, c->packet_index + done);
            if ((rc = scan_floor_kinds(ctx, io, c->packet_index * C, (c->packet_index + done) * C, &need_dense))) return rc;
        }
    }
    if (need_dense && !io->dense_floor) return fail(ctx, LWB_ERR_INVALID, "dense_floor missing");
    if (n_launch) {
        const bool host = io->memory == LWB_MEM_HOST;
        const float *d_coeffs = io->coeffs, *d_dense = io->dense_floor;
        char *d_pcm = (char *)io->pcm;
        cudaStream_t sm = ctx->stream;
        if (host) {
            // arenas are addressed with the caller's element offsets: bias the device pointers instead of the descriptors
            if ((rc = ensure(ctx, ctx->coeffs, (size_t)(c_hi - c_lo) * 4))) return rc;
            if (o_hi > o_lo && (rc = ensure(ctx, ctx->pcm, (size_t)(o_hi - o_lo) * esz))) return rc;
            CU(ctx, cudaMemcpyAsync(ctx->coeffs.p, io->coeffs + c_lo, (size_t)(c_hi - c_lo) * 4, cudaMemcpyHostToDevice, sm));
            d_coeffs = (const float *)ctx->coeffs.p - c_lo;
            if (need_dense) {
                if ((rc = ensure(ctx, ctx->dense, (size_t)(c_hi - c_lo) * 4))) return rc;
                CU(ctx, cudaMemcpyAsync(ctx->dense.p, io->dense_floor + c_lo, (size_t)(c_hi - c_lo) * 4, cudaMemcpyHostToDevice, sm));
                d_dense = (const float *)ctx->dense.p - c_lo;
            }
            d_pcm = (char *)ctx->pcm.p - o_lo * esz;
        }
        const uint8_t *d_kinds = nullptr;
        const uint32_t *d_ys = nullptr;
        if (residue && (rc = stage_floor_arrays(ctx, io, r_lo, r_hi, (unsigned)uniform_c, sm, &d_kinds, &d_ys))) return rc;
        // descriptors and mode bytes share one device buffer; a prepared batch (device memory, spectrum
        // entry) owns it and replays the launch while no stream changes shape
        const bool capture = plan && !host && !residue;
        DevBuf &dbuf = capture ? plan->mix : ctx->cdesc;
        const size_t used_desc = n_launch * sizeof(ChainDesc);
        if ((rc = ensure(ctx, dbuf, used_desc + boff + 16))) return rc;
        CU(ctx, cudaMemcpyAsync(dbuf.p, hd, used_desc, cudaMemcpyHostToDevice, sm));
        CU(ctx, cudaMemcpyAsync((char *)dbuf.p + used_desc, hb, boff + 16, cudaMemcpyHostToDevice, sm));
        CU(ctx, cudaEventRecord(st->ev, sm));
        st->pending = true;
        MixLaunch ml;
        ml.db = (char *)dbuf.p; ml.off_sr = 0; ml.off_cd = 0; ml.off_rc = 0; ml.off_sg = 0; ml.off_by = used_desc; ml.pack = nullptr; ml.spack = nullptr; ml.w_short = nullptr; ml.mpack = nullptr; ml.mid_kb = 0; ml.ls = 0;
        ml.i16 = false; ml.residue = residue; ml.out_format = io->out_format; ml.warps = maxc * wpc; ml.smem = smem;
        ml.n1max = n1max; ml.wpc = wpc; ml.np = np; ml.coeffs = d_coeffs; ml.dense = d_dense; ml.kinds = d_kinds; ml.ys = d_ys; ml.pcm = d_pcm;
        std::vector<MixRound> rounds(1, MixRound{0, 0, 0, 0, 0, n_launch});
        if ((rc = mixed_launch_rounds(ctx, ml, rounds))) return rc;
        if (capture) {
            plan->mixed_captured = true;
            plan->gen = gen_at_entry;
            plan->mix_launch = ml;
            plan->mix_rounds = std::move(rounds);
        }
        if (host) {
            if (o_hi > o_lo)
                CU(ctx, cudaMemcpyAsync((char *)io->pcm + o_lo * esz, ctx->pcm.p, (size_t)(o_hi - o_lo) * esz, cudaMemcpyDeviceToHost, sm));
            CU(ctx, cudaStreamSynchronize(sm));
        }
    }
    for (auto &e : ends)
        if (e.touched) set_stream_state(e.s, e.has, e.plen);
    return LWB_OK;
}

