// path_long.cuh -- part of the C-ABI translation unit (included by lwb_api.cu, not compiled on its own):
// the fused long-block path (kernel_long.cuh): run cutting, descriptor staging, host-memory chunk pipeline.
#pragma once

// ---------------------------------------------------------------------------------------------
// Fused path (kernel_long.cuh).  Eligible batches: spectrum entry, f32 or i16 out (planar, or interleaved with one
// channel count of at most 8 per batch), every packet a
// long block of blocksize 2^11 with long neighbours, every stream either empty or holding a
// 1024-sample right half.  Planned directly from the chain list in O(chains + mode bytes) -- at
// 0.8 G blocks/s per GPU a per-packet host plan would be the bottleneck.
// ---------------------------------------------------------------------------------------------
struct LongItem {
    lwb_chain *c;
    uint32_t P;
    bool has_prev;
};

static int acquire_staging(lwb_ctx *ctx, size_t bytes, Staging **out)
{
    Staging &st = ctx->stage[ctx->stage_next];
    ctx->stage_next = (ctx->stage_next + 1) % 3;
    if (!st.ev) CU(ctx, cudaEventCreateWithFlags(&st.ev, cudaEventDisableTiming));
    if (st.pending) {
        CU(ctx, cudaEventSynchronize(st.ev));      // waits for the descriptor copy only, not for kernels
        st.pending = false;
    }
    if (st.cap < bytes) {
        if (st.h) cudaFreeHost(st.h);
        st.h = nullptr;
        st.cap = 0;
        CU(ctx, cudaHostAlloc(&st.h, bytes * 2 + 4096, cudaHostAllocDefault));
        st.cap = bytes * 2 + 4096;
    }
    *out = &st;
    return LWB_OK;
}

// Whether k_long takes the batch's interleaved output at all (read once per call).  Not with LWB_NO_ITL set, and not
// for host-memory batches: their sliced H2D / kernel / D2H pipeline measured slower than the chain kernel's single
// pass for interleaved i16 residue batches (DESIGN 4.7), so those keep the chain kernel.
static bool long_takes_itl(const lwb_batch_io *io)
{
    return io->memory == LWB_MEM_DEVICE && !getenv("LWB_NO_ITL");
}

// PCM step of a channel on the fused kernels: 1 for planar output, C for interleaved output (k_long is instantiated
// for C <= 8; mono interleaved is the planar layout).  0: the batch's format stays off the fused kernels (interleaved
// output with more than 8 channels, or !itl_ok): the chain kernel writes it, as before k_long took interleaved output.
static unsigned long_step(int fmt, unsigned C, bool itl_ok)
{
    if (is_planar(fmt)) return 1;
    if (C > 8 || !itl_ok) return 0;
    return C;
}

// One past the last PCM element a chain of C channels writes.
static uint64_t pcm_end(const lwb_chain *c, unsigned C, bool planar, uint64_t n_samples)
{
    return c->out_offset + (planar ? (uint64_t)(C - 1) * c->out_stride + n_samples : n_samples * C);
}

// Appends the runs of one chain.  A chain (one channel of one stream) is cut into several runs
// when there are too few chains to fill the machine; every run after the first re-transforms the
// packet before its first one as a primer (its right half is all the run needs), which keeps
// runs independent at the cost of one extra IMDCT per cut.
// Planar output (step 1): a channel's runs one after the other.  Interleaved output (step C): cut by cut, the C runs
// that write one stretch of frames next to each other, so that the warps drawing them fill the same PCM lines at
// about the same time.
static void long_runs_of(const LongItem &it, size_t cuts, const float *coeffs, uint64_t coeff_base, char *pcm,
                         uint64_t pcm_base, size_t esz, unsigned step, LongRun *&w)
{
    const lwb_stream *s = it.c->stream;
    const lwb_setup *su = s->setup;
    const unsigned C = su->channels;
    const size_t P = it.P;
    const bool itl = step != 1;
    for (size_t q = 0; q < (size_t)C * cuts; q++) {
        const unsigned ch = (unsigned)(itl ? q % C : q / cuts);
        const size_t k = itl ? q / C : q % cuts;
        const float *in0 = coeffs + (it.c->coeff_offset - coeff_base) + (size_t)ch * kLongN2;
        char *out0 = pcm + ((it.c->out_offset - pcm_base) + (itl ? (size_t)ch : (size_t)ch * it.c->out_stride)) * esz;
        const size_t p0 = P * k / cuts, p1 = P * (k + 1) / cuts;   // this run emits packets [p0, p1)
        LongRun &r = *w++;
        std::memset(&r, 0, sizeof(r));
        r.in_stride = (uint32_t)(C * kLongN2);
        r.state = s->d_state + (size_t)ch * state_stride(su);
        r.write_state = (k + 1 == cuts);
        if (k == 0) {
            r.in = in0;
            r.n_packets = (uint32_t)(p1 - p0);
            r.has_prev = it.has_prev;
            r.out = out0;
        } else {
            r.in = in0 + (p0 - 1) * (size_t)r.in_stride;           // primer = packet p0 - 1
            r.n_packets = (uint32_t)(p1 - p0 + 1);
            r.has_prev = 0;
            // samples emitted before packet p0: packets 0..p0-1, minus the first if no state
            r.out = out0 + (size_t)(p0 - (it.has_prev ? 0 : 1)) * kLongN2 * step * esz;
        }
    }
}

// Every packet a long block of the fast blocksize with long neighbours, every stream empty or
// holding a 1024-sample right half, arenas aligned: what the fused kernel takes.
static bool batch_is_uniform_long(lwb_ctx *ctx, const lwb_chain *chains, size_t n_chains, const lwb_batch_io *io)
{
    const bool planar = is_planar(io->out_format);
    const bool itl_ok = long_takes_itl(io);
    const float *pack = nullptr;
    for (size_t i = 0; i < n_chains; i++) {
        const lwb_chain *c = &chains[i];
        if (!c->stream || c->stream->ctx != ctx || (c->n_packets && !c->mode_numbers)) return false;
        const lwb_stream *s = c->stream;
        const lwb_setup *su = s->setup;
        if (su->bs1 != kLongBs || !su->host.tab[1].pack) return false;
        if (pack && pack != su->host.tab[1].pack) return false;
        pack = su->host.tab[1].pack;
        if (!long_step(io->out_format, su->channels, itl_ok)) return false;
        if ((c->out_offset & 3) || (planar && (c->out_stride & 3)) || (c->coeff_offset & 3)) return false;
        if (s->has && s->plen != (uint32_t)kLongN2) return false;
        for (uint32_t k = 0; k < c->n_packets; k++) {
            const uint8_t m = c->mode_numbers[k];
            if (m >= su->n_modes || !su->host.mode_blockflag[m]) return false;
            if (c->prev_window_flags && !c->prev_window_flags[k]) return false;
            if (c->next_window_flags && !c->next_window_flags[k]) return false;
        }
    }
    return true;
}

// `spectrum_dev`: when non-null the spectrum has already been formed on the device (residue entry:
// k_prologue wrote it to ctx->spec, element offset `spectrum_base` = its [0]); the input side of the
// batch is then neither validated as a spectrum entry nor copied.
// Host-memory pipeline of the residue entries (try_long_residue): the caller has cut the batch into slices of chains
// and runs try_long once per slice; the PCM staging covers the whole batch, nothing is synchronised per slice.
struct LongSlice {
    bool active = false;
    uint64_t o_lo = 0, o_hi = 0;       // PCM element range of the whole batch (staging base)
    int ev_slot = 0;                   // which ev_done[] entry orders this slice's D2H
};

static int try_long(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io, uint64_t epoch,
                    bool *handled, const float *spectrum_dev = nullptr, uint64_t spectrum_base = 0,
                    lwb_plan *plan = nullptr, bool capture_with_spectrum_dev = false, LongSlice slice = LongSlice())
{
    *handled = false;
    const uint64_t gen_at_entry = ctx->state_gen;
    if (plan) plan->captured = false;
    if (!spectrum_dev && io->entry != LWB_ENTRY_SPECTRUM) return LWB_OK;
    if (getenv("LWB_FORCE_GENERIC")) return LWB_OK;
    const bool planar = is_planar(io->out_format);
    const bool i16 = io->out_format == LWB_OUT_I16_PLANAR || io->out_format == LWB_OUT_I16_INTERLEAVED;
    const size_t esz = elem_size(io->out_format);
    std::vector<LongItem> items;
    items.reserve(n_chains);
    const float *pack = nullptr;
    size_t chan_chains = 0;
    unsigned step = 0;                 // interleaved: one channel count per launch, it is the kernel's store step
    const bool itl_ok = long_takes_itl(io);
    for (size_t i = 0; i < n_chains; i++) {
        lwb_chain *c = &chains[i];
        if (!c->stream || c->stream->ctx != ctx || (c->n_packets && !c->mode_numbers)) return LWB_OK;   // generic path reports it
        const lwb_stream *s = c->stream;
        const lwb_setup *su = s->setup;
        if (su->bs1 != kLongBs || !su->host.tab[1].pack) return LWB_OK;
        if (pack && pack != su->host.tab[1].pack) return LWB_OK;          // one twiddle pack per launch
        pack = su->host.tab[1].pack;
        const unsigned cs = long_step(io->out_format, su->channels, itl_ok);
        if (!cs || (step && cs != step)) return LWB_OK;
        step = cs;
        if ((c->out_offset & 3) || (planar && (c->out_stride & 3)) || (c->coeff_offset & 3)) return LWB_OK;
        if (s->has && s->plen != (uint32_t)kLongN2) return LWB_OK;
        const uint32_t P = c->n_packets;
        for (uint32_t k = 0; k < P; k++) {
            const uint8_t m = c->mode_numbers[k];
            if (m >= su->n_modes || !su->host.mode_blockflag[m]) return LWB_OK;
            if (c->prev_window_flags && !c->prev_window_flags[k]) return LWB_OK;
            if (c->next_window_flags && !c->next_window_flags[k]) return LWB_OK;
        }
        items.push_back(LongItem{c, P, s->has});
        if (P) chan_chains += su->channels;
    }
    *handled = true;
    // from here on this path owns the batch
    uint64_t c_lo = ~0ull, c_hi = 0, o_lo = ~0ull, o_hi = 0;
    for (auto &it : items) {
        lwb_chain *c = it.c;
        if (!spectrum_dev) {       // (the residue path has already run this check while planning)
            if (c->stream->busy_epoch == epoch) return fail(ctx, LWB_ERR_INVALID, "a stream appears in two chains of one batch");
            c->stream->busy_epoch = epoch;
        }
        const unsigned C = c->stream->setup->channels;
        c->status = LWB_OK;
        c->packets_done = it.P;
        c->n_samples = it.P ? (uint32_t)((it.P - (it.has_prev ? 0 : 1)) * kLongN2) : 0;
        if (!it.P) continue;
        if (planar && c->out_stride < c->n_samples) return fail(ctx, LWB_ERR_BUFFER, "chain: out_stride smaller than the samples produced");
        c_lo = std::min(c_lo, c->coeff_offset);
        c_hi = std::max(c_hi, c->coeff_offset + (uint64_t)it.P * C * kLongN2);
        o_lo = std::min(o_lo, c->out_offset);
        o_hi = std::max(o_hi, pcm_end(c, C, planar, c->n_samples));
    }
    if (!chan_chains) return LWB_OK;
    const size_t warp_slots = (size_t)ctx->sm_count * kLongWarps * kLongNB;
    size_t target_runs = warp_slots * 4;                   // ~4 groups per warp evens out the tail
    if (const char *e = getenv("LWB_LONG_TARGET_RUNS")) target_runs = (size_t)atol(e);
    const size_t min_run = 8;                              // packets per run below which a cut costs > 12%
    int rc;
    constexpr uint32_t kTicketPool = 1024;
    if (!ctx->ticket.p) {
        if ((rc = ensure(ctx, ctx->ticket, kTicketPool * sizeof(unsigned int)))) return rc;
        for (int k = 0; k < 2; k++) {
            CU(ctx, cudaEventCreateWithFlags(&ctx->ev_desc[k], cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&ctx->ev_kdone[k], cudaEventDisableTiming));
        }
    }

    const bool host = io->memory == LWB_MEM_HOST;          // the pcm arena is in host memory
    const bool in_host = host && !spectrum_dev;            // ... and so is the coefficient arena
    // host memory: chunks of chains, H2D / kernel / D2H of consecutive chunks overlap on three streams
    size_t n_chunks = 1;
    if (host) {
        const size_t bytes = (size_t)(c_hi - c_lo) * 4;
        n_chunks = std::min<size_t>(std::max<size_t>(1, bytes >> 25), std::min<size_t>(8, items.size()));   // profiles/e2e_chunks_r1.log
        if (const char *e = getenv("LWB_E2E_CHUNKS")) n_chunks = std::max<size_t>(1, std::min<size_t>((size_t)atol(e), std::min<size_t>(64, items.size())));
        if (slice.active) n_chunks = 1;                    // the caller's slices are the chunks
    }
    const float *d_coeffs = spectrum_dev ? spectrum_dev : io->coeffs;
    char *d_pcm = (char *)io->pcm;
    uint64_t cbase = spectrum_dev ? spectrum_base : 0, obase = 0;
    if (host) {
        if (in_host) {
            if ((rc = ensure(ctx, ctx->coeffs, (size_t)(c_hi - c_lo) * 4))) return rc;
            d_coeffs = (const float *)ctx->coeffs.p;
            cbase = c_lo;
        }
        if (slice.active) { o_lo = slice.o_lo; o_hi = slice.o_hi; }      // (already ensured by the caller)
        else if (o_hi > o_lo && (rc = ensure(ctx, ctx->pcm, (size_t)(o_hi - o_lo) * esz))) return rc;
        d_pcm = (char *)ctx->pcm.p;
        obase = o_lo;
        if (!ctx->ev_in[0])
            for (int k = 0; k < 65; k++) {
                if (k < 64) CU(ctx, cudaEventCreateWithFlags(&ctx->ev_in[k], cudaEventDisableTiming));
                CU(ctx, cudaEventCreateWithFlags(&ctx->ev_done[k], cudaEventDisableTiming));
            }
        // the copy streams must not run ahead of work already queued on the compute stream that
        // still reads/writes the arenas (previous call): order them behind it
        if (!slice.active) {
            CU(ctx, cudaEventRecord(ctx->ev_done[64], ctx->stream));
            CU(ctx, cudaStreamWaitEvent(ctx->copy_in, ctx->ev_done[64], 0));
        }
    }
    // count runs
    std::vector<size_t> cuts(items.size(), 1);
    size_t total_runs = 0;
    for (size_t i = 0; i < items.size(); i++) {
        if (!items[i].P) { cuts[i] = 0; continue; }
        // per launch (chunk) the machine should see >= target_runs runs
        const size_t per_launch = std::max<size_t>(1, chan_chains / n_chunks);
        size_t k = 1;
        if (per_launch < target_runs) k = (target_runs + per_launch - 1) / per_launch;
        cuts[i] = std::max<size_t>(1, std::min(k, items[i].P / min_run));
        total_runs += cuts[i] * items[i].c->stream->setup->channels;
    }
    // the kernel takes groups of kLongNB runs of equal length; unpaired runs get a dummy partner
    const size_t cap_runs = total_runs * (kLongNB > 1 ? 2 : 1) + kLongNB;
    Staging *st;
    if ((rc = acquire_staging(ctx, cap_runs * sizeof(LongRun), &st))) return rc;
    const int par = ctx->runs_par;
    ctx->runs_par ^= 1;
    // a plan (device-memory batches) owns its descriptor buffer so that later executions can reuse it
    // (runs that read ctx->spec stay valid because growing any ctx arena bumps state_gen, see ensure())
    const bool capture = plan && !host && (!spectrum_dev || capture_with_spectrum_dev) && n_chunks == 1;
    DevBuf &rb = capture ? plan->runs : ctx->runs_buf[par];
    if ((rc = ensure(ctx, rb, cap_runs * sizeof(LongRun)))) return rc;
    LongRun *const d_runs_base = (LongRun *)rb.p;
    LongRun *h_runs = (LongRun *)st->h, *w = h_runs;
    std::vector<LongRun> tmp;
    struct ChunkPlan { size_t r0, nr; uint64_t kc_lo, kc_hi, ko_lo, ko_hi; };
    std::vector<ChunkPlan> cplan;
    std::vector<uint32_t> order;
    for (size_t k = 0; k < n_chunks; k++) {
        const size_t i0 = items.size() * k / n_chunks, i1 = items.size() * (k + 1) / n_chunks;
        LongRun *w0 = w;
        uint64_t kc_lo = ~0ull, kc_hi = 0, ko_lo = ~0ull, ko_hi = 0;
        // NB == 1: descriptors are written straight into the pinned staging; otherwise into a scratch
        // vector that is regrouped below
        size_t chunk_runs = 0;
        for (size_t i = i0; i < i1; i++)
            if (items[i].P) chunk_runs += cuts[i] * items[i].c->stream->setup->channels;
        LongRun *gen = w;
        if (kLongNB > 1) {
            tmp.resize(chunk_runs);
            gen = tmp.data();
        }
        for (size_t i = i0; i < i1; i++) {
            if (!items[i].P) continue;
            long_runs_of(items[i], cuts[i], d_coeffs, cbase, d_pcm, obase, esz, step, gen);
            const lwb_chain *c = items[i].c;
            const unsigned C = c->stream->setup->channels;
            kc_lo = std::min(kc_lo, c->coeff_offset);
            kc_hi = std::max(kc_hi, c->coeff_offset + (uint64_t)items[i].P * C * kLongN2);
            ko_lo = std::min(ko_lo, c->out_offset);
            ko_hi = std::max(ko_hi, pcm_end(c, C, planar, c->n_samples));
        }
        if (!chunk_runs) continue;
        if (kLongNB == 1) {
            w = gen;
        } else {
            // group runs of equal packet count (consecutive channels of a stream already are)
            bool sorted = true;
            for (size_t i = 1; i < tmp.size() && sorted; i++) sorted = tmp[i].n_packets == tmp[0].n_packets;
            order.resize(tmp.size());
            for (uint32_t i = 0; i < order.size(); i++) order[i] = i;
            if (!sorted)
                std::stable_sort(order.begin(), order.end(),
                                 [&](uint32_t a, uint32_t b) { return tmp[a].n_packets < tmp[b].n_packets; });
            size_t i = 0;
            while (i < order.size()) {
                size_t j = i;
                while (j < order.size() && tmp[order[j]].n_packets == tmp[order[i]].n_packets) j++;
                for (size_t q = i; q < j; q++) *w++ = tmp[order[q]];
                size_t fill = (kLongNB - (j - i) % kLongNB) % kLongNB;
                while (fill--) {
                    LongRun d = tmp[order[j - 1]];       // reads valid memory, stores nothing
                    d.dummy = 1;
                    d.write_state = 0;
                    d.has_prev = 0;
                    *w++ = d;
                }
                i = j;
            }
        }
        cplan.push_back(ChunkPlan{(size_t)(w0 - h_runs), (size_t)(w - w0), kc_lo, kc_hi, ko_lo, ko_hi});
    }
    // one descriptor upload for the whole call, on the copy stream, behind the kernel that last read
    // this half of the double buffer
    const size_t all_runs = (size_t)(w - h_runs);
    if (!all_runs) return LWB_OK;
    // (slices of a pipelined host batch: on the H2D stream -- behind copy_out's PCM copies the next slice's kernels would wait
    // for the previous slice's D2H)
    cudaStream_t ds = slice.active ? ctx->copy_in : ctx->copy_out;
    CU(ctx, cudaStreamWaitEvent(ds, ctx->ev_kdone[par], 0));
    CU(ctx, cudaMemcpyAsync(d_runs_base, h_runs, all_runs * sizeof(LongRun), cudaMemcpyHostToDevice, ds));
    CU(ctx, cudaEventRecord(ctx->ev_desc[par], ds));
    CU(ctx, cudaEventRecord(st->ev, ds));
    st->pending = true;
    CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_desc[par], 0));
    for (size_t k = 0; k < cplan.size(); k++) {
        const ChunkPlan &cp = cplan[k];
        if (in_host) {
            CU(ctx, cudaMemcpyAsync((float *)ctx->coeffs.p + (cp.kc_lo - cbase), io->coeffs + cp.kc_lo,
                                    (size_t)(cp.kc_hi - cp.kc_lo) * 4, cudaMemcpyHostToDevice, ctx->copy_in));
            CU(ctx, cudaEventRecord(ctx->ev_in[k], ctx->copy_in));
            CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_in[k], 0));
        }
        if (ctx->ticket_next % kTicketPool == 0)
            CU(ctx, cudaMemsetAsync(ctx->ticket.p, 0, kTicketPool * sizeof(unsigned int), ctx->stream));
        unsigned int *ticket = (unsigned int *)ctx->ticket.p + (ctx->ticket_next++ % kTicketPool);
        if (long_launch(ctx->stream, d_runs_base + cp.r0, (uint32_t)(cp.nr / kLongNB), pack, ticket, ctx->sm_count, i16, nullptr, 0, (int)step))
            return fail(ctx, LWB_ERR_CUDA, "long kernel launch", cudaGetLastError());
        ctx->launches++;
        ctx->long_launches++;
        if (host && cp.ko_hi > cp.ko_lo) {
            const size_t evk = slice.active ? (size_t)slice.ev_slot : k;
            CU(ctx, cudaEventRecord(ctx->ev_done[evk], ctx->stream));
            CU(ctx, cudaStreamWaitEvent(ctx->copy_out, ctx->ev_done[evk], 0));
            CU(ctx, cudaMemcpyAsync((char *)io->pcm + cp.ko_lo * esz, (char *)ctx->pcm.p + (cp.ko_lo - obase) * esz,
                                    (size_t)(cp.ko_hi - cp.ko_lo) * esz, cudaMemcpyDeviceToHost, ctx->copy_out));
        }
    }
    CU(ctx, cudaEventRecord(ctx->ev_kdone[par], ctx->stream));
    if (capture && cplan.size() == 1) {
        plan->captured = true;
        plan->gen = gen_at_entry;          // valid while no stream changed shape since planning
        plan->n_groups = (uint32_t)(cplan[0].nr / kLongNB);
        plan->pack = pack;
        plan->i16 = i16;
        plan->step = (int)step;
    }
    if (host && !slice.active) {
        CU(ctx, cudaStreamSynchronize(ctx->copy_out));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    for (auto &it : items)
        if (it.P) set_stream_state(it.c->stream, true, kLongN2);
    return LWB_OK;
}

// Residue-entry batches whose every packet is a long block with long neighbours (what the fused
// kernel takes) -- decided from the generic plan.
static bool plan_is_long(const std::vector<PlanChain> &plan, const lwb_batch_io *io)
{
    if (getenv("LWB_FORCE_GENERIC")) return false;
    const bool itl_ok = long_takes_itl(io);
    for (auto &pc : plan) {
        const lwb_setup *su = pc.c->stream->setup;
        if (su->bs1 != kLongBs || !su->host.tab[1].pack) return false;
        if (!long_step(io->out_format, su->channels, itl_ok)) return false;
        if (pc.c->status != LWB_OK) return false;
        for (auto &pp : pc.pk) {
            if (!pp.g.blockflag || pp.g.ls != 0 || pp.g.rs != (pp.g.n >> 1) || pp.g.re != pp.g.n) return false;
            if (pp.plen != 0 && pp.plen != (pp.g.n >> 1)) return false;
        }
    }
    return true;
}

// k_prologue over every packet of the plan: ctx->spec[coeff_off] <- floor x decoupled residue.
static int run_prologue_all(lwb_ctx *ctx, std::vector<PlanChain> &plan, const DevArenas &ar, size_t spec_elems)
{
    size_t n_desc = 0;
    for (auto &pc : plan) n_desc += pc.pk.size();
    if (!n_desc) return LWB_OK;
    int rc;
    if ((rc = ensure_pinned(ctx, n_desc * sizeof(DevPacket)))) return rc;
    if ((rc = ensure(ctx, ctx->desc, n_desc * sizeof(DevPacket)))) return rc;
    if ((rc = ensure(ctx, ctx->spec, spec_elems * sizeof(float)))) return rc;
    CU(ctx, cudaStreamSynchronize(ctx->stream));          // pinned descriptor staging is reused
    DevPacket *hp = (DevPacket *)ctx->h_desc;
    size_t di = 0;
    for (auto &pc : plan) {
        const lwb_setup *su = pc.c->stream->setup;
        for (size_t k = 0; k < pc.pk.size(); k++) {
            const PlanPacket &pp = pc.pk[k];
            DevPacket &d = hp[di++];
            std::memset(&d, 0, sizeof(d));
            d.setup = su->d_setup;
            d.coeff_off = pp.coeff_off - ar.coeff_base;
            d.pkt_index = pc.c->packet_index + k - ar.kinds_row0;
            d.n = (uint16_t)pp.g.n;
            d.blockflag = pp.g.blockflag;
            d.mapping = pp.g.mapping;
            d.channels = su->channels;
        }
    }
    CU(ctx, cudaMemcpyAsync(ctx->desc.p, hp, n_desc * sizeof(DevPacket), cudaMemcpyHostToDevice, ctx->stream));
    return launch_prologue(ctx, (const DevPacket *)ctx->desc.p, hp, n_desc, plan[0].c->stream->setup->channels, prologue_smem_of(plan),
                           ar.coeffs, ar.dense, ar.kinds, ar.ys, (float *)ctx->spec.p, ar.vq);
}


// Residue-entry batches whose every packet is a long block with long neighbours: the front stages
// (k_floor1_segments + k_prologue_fused, or k_prologue) form the spectrum on the device, the fused kernel does the
// rest.  Planned straight from the chain list like try_long (no per-packet PlanChain vectors); a prepared batch
// keeps the front-stage descriptors and, for device-memory batches, the fused kernel's runs, so that a replay
// is three launches with no host work (lwb_plan_execute).
static int try_long_residue(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io, uint64_t epoch, bool *handled,
                            lwb_plan *plan)
{
    *handled = false;
    if (io->entry == LWB_ENTRY_SPECTRUM || getenv("LWB_FORCE_GENERIC")) return LWB_OK;
    if (!batch_is_uniform_long(ctx, chains, n_chains, io)) return LWB_OK;
    const bool vq = io->entry == LWB_ENTRY_VQ;
    if (!io->floor_kind) return fail(ctx, LWB_ERR_INVALID, "residue entry needs floor_kind");
    unsigned C = 0;
    size_t n_pk = 0;
    uint64_t c_lo = ~0ull, c_hi = 0, r_lo = ~0ull, r_hi = 0;
    bool need_dense = false;
    int rc;
    for (size_t i = 0; i < n_chains; i++) {
        const lwb_chain *c = &chains[i];
        const unsigned cc = c->stream->setup->channels;
        if (!C) C = cc;
        if (C != cc) return fail(ctx, LWB_ERR_INVALID, "residue batches need one channel count");
        if (!c->n_packets) continue;
        n_pk += c->n_packets;
        c_lo = std::min(c_lo, c->coeff_offset);
        c_hi = std::max(c_hi, c->coeff_offset + (uint64_t)c->n_packets * C * kLongN2);
        r_lo = std::min(r_lo, c->packet_index);
        r_hi = std::max<uint64_t>(r_hi, c->packet_index + c->n_packets);
        if ((rc = scan_floor_kinds(ctx, io, c->packet_index * C, (c->packet_index + c->n_packets) * C, &need_dense))) return rc;
    }
    if (need_dense && !io->dense_floor) return fail(ctx, LWB_ERR_INVALID, "dense_floor missing");
    for (size_t i = 0; i < n_chains; i++) {
        lwb_stream *s = chains[i].stream;
        if (s->busy_epoch == epoch) return fail(ctx, LWB_ERR_INVALID, "a stream appears in two chains of one batch");
        s->busy_epoch = epoch;
    }
    *handled = true;
    if (!n_pk) {
        for (size_t i = 0; i < n_chains; i++) { chains[i].status = LWB_OK; chains[i].packets_done = 0; chains[i].n_samples = 0; }
        return LWB_OK;
    }
    cudaStream_t sm = ctx->stream;
    const size_t elems = (size_t)(c_hi - c_lo);
    const bool host = io->memory == LWB_MEM_HOST;
    const float *d_res = vq ? nullptr : io->coeffs, *d_dense = need_dense ? io->dense_floor : nullptr;
    if (host) {
        if (!vq) {
            if ((rc = ensure(ctx, ctx->coeffs, elems * 4))) return rc;
            d_res = (const float *)ctx->coeffs.p - c_lo;
        }
        if (need_dense) {
            if ((rc = ensure(ctx, ctx->dense, elems * 4))) return rc;
            d_dense = (const float *)ctx->dense.p - c_lo;
        }
    }
    if ((rc = ensure(ctx, ctx->spec, elems * 4))) return rc;
    float *d_spec = (float *)ctx->spec.p - c_lo;
    // front-stage descriptors: absolute element offsets and packet rows (the arena pointers are biased instead)
    const DevPacket *d_pk;
    bool fast;
    const size_t smem_old = prologue_smem((int)C, kLongBs);
    if (plan && plan->pro_captured && plan->n_pro == n_pk) {
        d_pk = (const DevPacket *)plan->pro.p;
        fast = plan->pro_fast;
    } else {
        Staging *st;
        if ((rc = acquire_staging(ctx, n_pk * sizeof(DevPacket), &st))) return rc;
        DevBuf &db = plan ? plan->pro : ctx->desc;
        if ((rc = ensure(ctx, db, n_pk * sizeof(DevPacket)))) return rc;
        DevPacket *hp = (DevPacket *)st->h;
        size_t di = 0;
        for (size_t i = 0; i < n_chains; i++) {
            const lwb_chain *c = &chains[i];
            const lwb_setup *su = c->stream->setup;
            for (uint32_t k = 0; k < c->n_packets; k++) {
                DevPacket &d = hp[di++];
                std::memset(&d, 0, sizeof(d));
                d.setup = su->d_setup;
                d.coeff_off = c->coeff_offset + (uint64_t)k * C * kLongN2;
                d.pkt_index = c->packet_index + k;
                d.n = kLongN;
                d.blockflag = 1;
                d.mapping = su->host.mode_mapping[c->mode_numbers[k]];
                d.channels = (uint8_t)C;
            }
        }
        fast = prologue_is_fast(hp, n_pk, C, d_res, d_dense, d_spec);
        CU(ctx, cudaMemcpyAsync(db.p, hp, n_pk * sizeof(DevPacket), cudaMemcpyHostToDevice, sm));
        CU(ctx, cudaEventRecord(st->ev, sm));
        st->pending = true;
        d_pk = (const DevPacket *)db.p;
        if (plan) {
            plan->pro_captured = true;
            plan->pro_fast = fast;
            plan->n_pro = n_pk;
            plan->pro_smem_old = smem_old;
            plan->pro_C = C;
            plan->pro_c_lo = c_lo; plan->pro_c_hi = c_hi; plan->pro_r_lo = r_lo; plan->pro_r_hi = r_hi;
        }
    }
    if (!host) {
        const uint8_t *d_kinds;
        const uint32_t *d_ys;
        if ((rc = stage_floor_arrays(ctx, io, r_lo, r_hi, C, sm, &d_kinds, &d_ys))) return rc;
        VqView vqv;
        if ((rc = stage_vq_arrays(ctx, io, r_lo, r_hi, sm, &vqv))) return rc;
        if ((rc = launch_prologue(ctx, d_pk, n_pk, C, fast, smem_old, kLongN2, d_res, d_dense, d_kinds, d_ys, d_spec, vqv))) return rc;
        bool h2 = false;
        rc = try_long(ctx, chains, n_chains, io, epoch, &h2, (const float *)ctx->spec.p, c_lo, plan, true);
        if (rc) return rc;
        if (!h2) return fail(ctx, LWB_ERR_INVALID, "internal: uniform long residue batch refused by the fused path");
        return LWB_OK;
    }
    // Host memory: slices of chains flow through three streams -- copy_in brings a slice's inputs (dense residues, or
    // VQ runs / entries, and its floor rows), the compute stream runs its front stages and the fused kernel, copy_out
    // takes its PCM home -- so that H2D, kernels and D2H of consecutive slices overlap (the link is duplex).
    size_t n_sl = std::min<size_t>(std::max<size_t>(1, (n_pk * (size_t)C * kLongN2 * 4) >> 25), std::min<size_t>(8, n_chains));
    if (const char *e = getenv("LWB_E2E_CHUNKS")) n_sl = std::max<size_t>(1, std::min<size_t>((size_t)atol(e), std::min<size_t>(32, n_chains)));
    // whole-batch staging (absolute rows / offsets address it); each slice copies its own part
    const size_t esz = elem_size(io->out_format);
    const bool planar = is_planar(io->out_format);
    uint64_t o_lo = ~0ull, o_hi = 0;
    for (size_t i = 0; i < n_chains; i++) {
        const lwb_chain *c = &chains[i];
        if (!c->n_packets) continue;
        const uint64_t ns = (uint64_t)(c->n_packets - (c->stream->has ? 0 : 1)) * kLongN2;
        o_lo = std::min(o_lo, c->out_offset);
        o_hi = std::max(o_hi, pcm_end(c, C, planar, ns));
    }
    if (o_hi > o_lo && (rc = ensure(ctx, ctx->pcm, (size_t)(o_hi - o_lo) * esz))) return rc;
    const bool host_floors = io->floor_memory != LWB_MEM_DEVICE;
    const size_t rows_all = (size_t)(r_hi - r_lo) * C;
    VqView vqv;
    const uint8_t *d_kinds = io->floor_kind;
    const uint32_t *d_ys = io->floor1_y;
    uint64_t vo_lo = 0, ve_lo = 0;
    if (host_floors) {
        if ((rc = ensure(ctx, ctx->kinds, rows_all)) || (io->floor1_y && (rc = ensure(ctx, ctx->ys, rows_all * LWB_MAX_POSTS * sizeof(uint32_t))))) return rc;
        d_kinds = (const uint8_t *)ctx->kinds.p - r_lo * C;
        d_ys = io->floor1_y ? (const uint32_t *)ctx->ys.p - r_lo * C * LWB_MAX_POSTS : nullptr;
        if (vq) {
            vo_lo = io->vq_run_offsets[r_lo];
            ve_lo = io->vq_entry_offsets[r_lo];
            const uint64_t vo_hi = io->vq_run_offsets[r_hi], ve_hi = io->vq_entry_offsets[r_hi];
            if (vo_hi < vo_lo || ve_hi < ve_lo) return fail(ctx, LWB_ERR_INVALID, "vq offsets must be non-decreasing");
            const size_t b_off = ((size_t)(r_hi - r_lo) + 1) * sizeof(uint64_t), b_run = std::max<size_t>((size_t)(vo_hi - vo_lo), 1) * sizeof(lwb_vq_run);
            if ((rc = ensure(ctx, ctx->vqoff, 2 * b_off)) ||
                (rc = ensure(ctx, ctx->vqrec, b_run + std::max<size_t>((size_t)(ve_hi - ve_lo), 1) * sizeof(uint16_t) + 16)))
                return rc;
            vqv.run_off = (const uint64_t *)ctx->vqoff.p - r_lo;
            vqv.ent_off = (const uint64_t *)((char *)ctx->vqoff.p + b_off) - r_lo;
            vqv.runs = (const lwb_vq_run *)ctx->vqrec.p - vo_lo;
            vqv.entries = (const uint16_t *)((char *)ctx->vqrec.p + b_run) - ve_lo;
        }
    } else if ((rc = stage_vq_arrays(ctx, io, r_lo, r_hi, sm, &vqv))) {
        return rc;
    }
    if (!ctx->ev_in[0])
        for (int k = 0; k < 65; k++) {
            if (k < 64) CU(ctx, cudaEventCreateWithFlags(&ctx->ev_in[k], cudaEventDisableTiming));
            CU(ctx, cudaEventCreateWithFlags(&ctx->ev_done[k], cudaEventDisableTiming));
        }
    // the copy streams must not run ahead of work already queued on the compute stream (previous call, descriptor upload)
    CU(ctx, cudaEventRecord(ctx->ev_done[64], sm));
    CU(ctx, cudaStreamWaitEvent(ctx->copy_in, ctx->ev_done[64], 0));
    CU(ctx, cudaStreamWaitEvent(ctx->copy_out, ctx->ev_done[64], 0));
    size_t pk0 = 0;
    for (size_t sl = 0; sl < n_sl; sl++) {
        const size_t i0 = n_chains * sl / n_sl, i1 = n_chains * (sl + 1) / n_sl;
        uint64_t sc_lo = ~0ull, sc_hi = 0, sr_lo = ~0ull, sr_hi = 0;
        size_t npk_sl = 0;
        for (size_t i = i0; i < i1; i++) {
            const lwb_chain *c = &chains[i];
            if (!c->n_packets) continue;
            npk_sl += c->n_packets;
            sc_lo = std::min(sc_lo, c->coeff_offset);
            sc_hi = std::max(sc_hi, c->coeff_offset + (uint64_t)c->n_packets * C * kLongN2);
            sr_lo = std::min(sr_lo, c->packet_index);
            sr_hi = std::max<uint64_t>(sr_hi, c->packet_index + c->n_packets);
        }
        if (!npk_sl) continue;
        cudaStream_t ci = ctx->copy_in;
        if (!vq)
            CU(ctx, cudaMemcpyAsync((float *)ctx->coeffs.p + (sc_lo - c_lo), io->coeffs + sc_lo, (size_t)(sc_hi - sc_lo) * 4, cudaMemcpyHostToDevice, ci));
        if (need_dense)
            CU(ctx, cudaMemcpyAsync((float *)ctx->dense.p + (sc_lo - c_lo), io->dense_floor + sc_lo, (size_t)(sc_hi - sc_lo) * 4, cudaMemcpyHostToDevice, ci));
        if (host_floors) {
            const size_t rr = (size_t)(sr_hi - sr_lo) * C;
            CU(ctx, cudaMemcpyAsync((uint8_t *)ctx->kinds.p + (sr_lo - r_lo) * C, io->floor_kind + sr_lo * C, rr, cudaMemcpyHostToDevice, ci));
            if (io->floor1_y)
                CU(ctx, cudaMemcpyAsync((uint32_t *)ctx->ys.p + (sr_lo - r_lo) * C * LWB_MAX_POSTS, io->floor1_y + sr_lo * C * LWB_MAX_POSTS,
                                        rr * LWB_MAX_POSTS * sizeof(uint32_t), cudaMemcpyHostToDevice, ci));
            if (vq) {
                const uint64_t a = io->vq_run_offsets[sr_lo], b = io->vq_run_offsets[sr_hi], ea = io->vq_entry_offsets[sr_lo], eb = io->vq_entry_offsets[sr_hi];
                const size_t nrow = (size_t)(sr_hi - sr_lo) + 1;
                CU(ctx, cudaMemcpyAsync(const_cast<uint64_t *>(vqv.run_off) + sr_lo, io->vq_run_offsets + sr_lo, nrow * 8, cudaMemcpyHostToDevice, ci));
                CU(ctx, cudaMemcpyAsync(const_cast<uint64_t *>(vqv.ent_off) + sr_lo, io->vq_entry_offsets + sr_lo, nrow * 8, cudaMemcpyHostToDevice, ci));
                if (b > a) CU(ctx, cudaMemcpyAsync(const_cast<lwb_vq_run *>(vqv.runs) + a, io->vq_runs + a, (size_t)(b - a) * sizeof(lwb_vq_run), cudaMemcpyHostToDevice, ci));
                if (eb > ea) CU(ctx, cudaMemcpyAsync(const_cast<uint16_t *>(vqv.entries) + ea, io->vq_entries + ea, (size_t)(eb - ea) * 2, cudaMemcpyHostToDevice, ci));
            }
        }
        CU(ctx, cudaEventRecord(ctx->ev_in[sl], ci));
        CU(ctx, cudaStreamWaitEvent(sm, ctx->ev_in[sl], 0));
        if ((rc = launch_prologue(ctx, d_pk + pk0, npk_sl, C, fast, smem_old, kLongN2, d_res, d_dense, d_kinds, d_ys, d_spec, vqv))) return rc;
        pk0 += npk_sl;
        bool h2 = false;
        LongSlice ls;
        ls.active = true;
        ls.o_lo = o_lo;
        ls.o_hi = o_hi;
        ls.ev_slot = (int)sl;
        rc = try_long(ctx, chains + i0, i1 - i0, io, epoch, &h2, (const float *)ctx->spec.p, c_lo, nullptr, false, ls);
        if (rc) return rc;
        if (!h2) return fail(ctx, LWB_ERR_INVALID, "internal: uniform long residue batch refused by the fused path");
    }
    CU(ctx, cudaStreamSynchronize(ctx->copy_out));
    CU(ctx, cudaStreamSynchronize(sm));
    return LWB_OK;
}
