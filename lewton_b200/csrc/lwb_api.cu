// lwb_api.cu -- the C ABI (include/lewton_b200.h): context, setup, stream state and batch
// submission.  Host logic mirrors the control flow of lewton's read_audio_packet_generic back
// half (src/audio.rs:988-1157): which window shape a packet has, whether a previous right half
// exists, what the packet returns -- all of that is decided here on the host from the mode bits
// (it never depends on sample values), so the kernels receive fully resolved descriptors and the
// device never has to be synchronised to learn a length.
#include <cuda_runtime.h>
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <new>
#include <string>
#include <vector>

#include "kernel_long.cuh"
#include "kernel_short.cuh"
#include "kernel_mid.cuh"
#include "kernels_generic.cuh"
#include "kernel_chain.cuh"
#include "kernel_prologue.cuh"
#include "lwb_common.h"

namespace lwb {
int generate_tables(int bs, float *a, float *b, float *c, float *window, uint32_t *bitrev);
int prepare_floor1(const lwb_floor_desc &d, DevFloor1 *out);
}  // namespace lwb

using namespace lwb;

#include "host_objects.cuh"

// ---------------------------------------------------------------------------------------------
// library / context
// ---------------------------------------------------------------------------------------------
extern "C" int lwb_abi_version(void) { return LWB_ABI_VERSION; }

extern "C" int lwb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int lwb_ctx_create(int device, lwb_ctx **out)
{
    if (!out) return LWB_ERR_INVALID;
    *out = nullptr;
    int n = lwb_device_count();
    if (n <= 0 || device < 0 || device >= n) return LWB_ERR_NO_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return LWB_ERR_NO_DEVICE;
    if (prop.major != 10) return LWB_ERR_NO_DEVICE;       // kernels are built for sm_100a only
    lwb_ctx *ctx = new (std::nothrow) lwb_ctx();
    if (!ctx) return LWB_ERR_BUFFER;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaSetDevice(device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return LWB_ERR_CUDA;
    }
    if (const char *e = getenv("LWB_SCRATCH_MB")) {
        long mb = atol(e);
        if (mb >= 1) ctx->x_cap_elems = (size_t)mb << 18;
    }
    long_kernel_configure();
    short_kernel_configure();
    mid_kernel_configure();
    prologue_kernel_configure();
    *out = ctx;
    return LWB_OK;
}

extern "C" void lwb_ctx_destroy(lwb_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (DevBuf *b : {&ctx->coeffs, &ctx->dense, &ctx->pcm, &ctx->spec, &ctx->segtab, &ctx->vqoff, &ctx->vqrec, &ctx->magic, &ctx->x, &ctx->desc,
                      &ctx->kinds, &ctx->ys, &ctx->chains, &ctx->ticket, &ctx->runs_buf[0], &ctx->runs_buf[1],
                      &ctx->cdesc, &ctx->cbytes})
        if (b->p) cudaFree(b->p);
    for (CachedTables &ct : ctx->tables)
        for (void *p : ct.allocs) cudaFree(p);
    if (ctx->h_desc) cudaFreeHost(ctx->h_desc);
    for (Staging &st : ctx->stage) {
        if (st.h) cudaFreeHost(st.h);
        if (st.ev) cudaEventDestroy(st.ev);
    }
    for (cudaEvent_t e : ctx->ev_in) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->ev_done) if (e) cudaEventDestroy(e);
    for (int k = 0; k < 2; k++) {
        if (ctx->ev_desc[k]) cudaEventDestroy(ctx->ev_desc[k]);
        if (ctx->ev_kdone[k]) cudaEventDestroy(ctx->ev_kdone[k]);
    }
    cudaStreamDestroy(ctx->stream);
    cudaStreamDestroy(ctx->copy_in);
    cudaStreamDestroy(ctx->copy_out);
    delete ctx;
}

extern "C" int lwb_ctx_synchronize(lwb_ctx *ctx)
{
    if (!ctx) return LWB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return LWB_OK;
}

extern "C" const char *lwb_last_error(const lwb_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }
extern "C" void *lwb_ctx_cuda_stream(lwb_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
extern "C" uint64_t lwb_ctx_launch_count(const lwb_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" uint64_t lwb_ctx_long_launch_count(const lwb_ctx *ctx) { return ctx ? ctx->long_launches : 0; }

extern "C" void *lwb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void lwb_host_free(void *p) { if (p) cudaFreeHost(p); }

// NUMA placement of the host side.  A rank that feeds GPU d through host buffers should run on, and
// allocate its pinned memory from, the socket GPU d's PCIe root hangs off: with 4 GPUs per socket the
// copies of all of them otherwise cross the inter-socket link of whichever node the pages landed on.
// Plain syscalls (no libnuma in this image).  Returns the node, or -1 when it cannot be determined.
extern "C" int lwb_bind_host_to_device(int device)
{
    if (device < 0) {
        syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
        return -1;
    }
    char busid[64] = {0};
    if (cudaDeviceGetPCIBusId(busid, (int)sizeof(busid) - 1, device) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    for (char *c = busid; *c; c++) *c = (char)tolower((unsigned char)*c);
    char path[160];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", busid);
    int node = -1;
    if (FILE *f = fopen(path, "r")) {
        if (fscanf(f, "%d", &node) != 1) node = -1;
        fclose(f);
    }
    if (node < 0 || node >= 1024) return -1;
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    cpu_set_t want, cur;
    CPU_ZERO(&want);
    if (FILE *f = fopen(path, "r")) {
        int a, b;
        while (fscanf(f, "%d", &a) == 1) {
            b = a;
            int ch = fgetc(f);
            if (ch == '-') {
                if (fscanf(f, "%d", &b) != 1) break;
                ch = fgetc(f);
            }
            for (int k = a; k <= b && k < CPU_SETSIZE; k++) CPU_SET(k, &want);
            if (ch != ',') break;
        }
        fclose(f);
    }
    if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {
        cpu_set_t both;
        CPU_AND(&both, &want, &cur);
        if (CPU_COUNT(&both) > 0) sched_setaffinity(0, sizeof(both), &both);
    }
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(sizeof(mask) * 8));
    return node;
}

extern "C" int lwb_device_alloc(lwb_ctx *ctx, size_t bytes, void **out)
{
    if (!ctx || !out) return LWB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMalloc(out, bytes ? bytes : 1));
    return LWB_OK;
}
extern "C" void lwb_device_free(lwb_ctx *ctx, void *p)
{
    if (!ctx || !p) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(p);
}
extern "C" int lwb_memcpy_h2d(lwb_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    if (!ctx) return LWB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return LWB_OK;
}
extern "C" int lwb_memcpy_d2h(lwb_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    if (!ctx) return LWB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return LWB_OK;
}

extern "C" int lwb_tables_generate(int bs, float *a, float *b, float *c, float *window, uint32_t *bitrev)
{
    return generate_tables(bs, a, b, c, window, bitrev);
}

// ---------------------------------------------------------------------------------------------
// setup
// ---------------------------------------------------------------------------------------------
template <typename T>
static int upload(lwb_setup *su, const T *host, size_t count, const T **dev)
{
    void *p = nullptr;
    lwb_ctx *ctx = su->ctx;
    CU(ctx, cudaMalloc(&p, std::max<size_t>(count * sizeof(T), 16)));
    su->allocs.push_back(p);
    if (count) CU(ctx, cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    *dev = (const T *)p;
    return LWB_OK;
}

extern "C" void lwb_setup_destroy(lwb_setup *su)
{
    if (!su) return;
    cudaSetDevice(su->ctx->device);
    cudaStreamSynchronize(su->ctx->stream);
    for (void *p : su->allocs) cudaFree(p);
    delete su;
}

extern "C" int lwb_setup_create(lwb_ctx *ctx, const lwb_setup_desc *d, lwb_setup **out)
{
    if (!ctx || !d || !out) return LWB_ERR_INVALID;
    *out = nullptr;
    // header.rs:239-243 (blocksizes, channels)
    if (d->blocksize_0 < 6 || d->blocksize_0 > 13 || d->blocksize_1 < 6 || d->blocksize_1 > 13 ||
        d->blocksize_0 > d->blocksize_1 || d->audio_channels == 0)
        return fail(ctx, LWB_ERR_BAD_FORMAT, "setup: blocksizes/channels out of range");
    if (d->n_modes == 0 || d->n_modes > LWB_MAX_MODES || d->n_mappings == 0 || d->n_mappings > 64 ||
        d->n_floors == 0 || d->n_floors > 64 || !d->modes || !d->mappings || !d->floors)
        return fail(ctx, LWB_ERR_INVALID, "setup: counts out of range");
    CU(ctx, cudaSetDevice(ctx->device));
    lwb_setup *su = new (std::nothrow) lwb_setup();
    if (!su) return LWB_ERR_BUFFER;
    su->ctx = ctx;
    su->channels = d->audio_channels;
    su->bs0 = d->blocksize_0;
    su->bs1 = d->blocksize_1;
    su->n_modes = d->n_modes;
    su->n_mappings = d->n_mappings;
    std::memset(&su->host, 0, sizeof(su->host));
    int rc = LWB_OK;
    // tables (header_cached.rs:33-41): the caller's own, or generated here
    for (int i = 0; i < 2 && rc == LWB_OK; i++) {
        const int bs = i ? d->blocksize_1 : d->blocksize_0;
        const size_t n = (size_t)1 << bs;
        std::vector<float> a(n / 2), b(n / 2), c(n / 4), w(n / 2);
        std::vector<uint32_t> br(n / 8);
        const lwb_tables_ref &t = d->tables[i];
        if (t.a) {
            if (!t.b || !t.c || !t.window || !t.bitrev) { rc = LWB_ERR_INVALID; break; }
            std::copy(t.a, t.a + n / 2, a.begin());
            std::copy(t.b, t.b + n / 2, b.begin());
            std::copy(t.c, t.c + n / 4, c.begin());
            std::copy(t.window, t.window + n / 2, w.begin());
            std::copy(t.bitrev, t.bitrev + n / 8, br.begin());
        } else {
            generate_tables(bs, a.data(), b.data(), c.data(), w.data(), br.data());
        }
        // Blocksize tables live in the context and are shared by every setup that has the same ones (bit for
        // bit): streams opened from different headers then still run in one launch of the fused kernels, which
        // take one twiddle pack per launch.
        const CachedTables *hit = nullptr;
        for (const CachedTables &ct : ctx->tables)
            if (ct.dt.bs == bs && ct.a == a && ct.b == b && ct.c == c && ct.w == w && ct.br == br) { hit = &ct; break; }
        if (!hit) {
            CachedTables ct;
            ct.dt.bs = bs;
            ct.dt.pad = 0;
            ct.dt.pack = nullptr;
            auto up = [&](const void *h, size_t bytes, const void **dev) {
                void *p = nullptr;
                if (cudaMalloc(&p, std::max<size_t>(bytes, 16)) != cudaSuccess) return LWB_ERR_CUDA;
                ct.allocs.push_back(p);
                if (cudaMemcpyAsync(p, h, bytes, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) return LWB_ERR_CUDA;
                *dev = p;
                return LWB_OK;
            };
            std::vector<float> pack;
            if (bs == kLongBs) {
                pack.resize(kLongPackFloats);
                long_build_pack(a.data(), b.data(), c.data(), w.data(), pack.data());
            } else if (bs == kShortBs) {
                pack.resize(kShortPackFloats);
                short_build_pack(a.data(), b.data(), c.data(), w.data(), pack.data());
            } else if (bs == 10) {
                pack.resize(kLongPackFloats);
                mid_build_pack<1>(a.data(), b.data(), c.data(), w.data(), pack.data());
            } else if (bs == 9) {
                pack.resize(kLongPackFloats);
                mid_build_pack<2>(a.data(), b.data(), c.data(), w.data(), pack.data());
            }
            rc = up(a.data(), a.size() * 4, (const void **)&ct.dt.a);
            if (!rc) rc = up(b.data(), b.size() * 4, (const void **)&ct.dt.b);
            if (!rc) rc = up(c.data(), c.size() * 4, (const void **)&ct.dt.c);
            if (!rc) rc = up(w.data(), w.size() * 4, (const void **)&ct.dt.window);
            if (!rc) rc = up(br.data(), br.size() * 4, (const void **)&ct.dt.bitrev);
            if (!rc && !pack.empty()) rc = up(pack.data(), pack.size() * 4, (const void **)&ct.dt.pack);
            // the copies above read from vectors that die here
            if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = LWB_ERR_CUDA;
            if (rc) {
                for (void *p : ct.allocs) cudaFree(p);
                fail(ctx, rc, "setup: table upload");
                break;
            }
            ct.a = a; ct.b = b; ct.c = c; ct.w = w; ct.br = br;
            ctx->tables.push_back(std::move(ct));
            hit = &ctx->tables.back();
        }
        su->host.tab[i] = hit->dt;
    }
    std::vector<DevFloor1> floors(d->n_floors);
    for (uint32_t i = 0; i < d->n_floors && rc == LWB_OK; i++) rc = prepare_floor1(d->floors[i], &floors[i]);
    su->mappings.resize(d->n_mappings);
    for (uint32_t i = 0; i < d->n_mappings && rc == LWB_OK; i++) {
        const lwb_mapping_desc &m = d->mappings[i];
        DevMapping &dm = su->mappings[i];
        std::memset(&dm, 0, sizeof(dm));
        if (m.coupling_steps > LWB_MAX_COUPLING || m.submaps == 0 || m.submaps > LWB_MAX_SUBMAPS) {
            rc = LWB_ERR_BAD_FORMAT;
            break;
        }
        dm.n_coupling = m.coupling_steps;
        for (int s = 0; s < m.coupling_steps; s++) {
            // header.rs:1006-1011
            if (m.magnitudes[s] == m.angles[s] || m.magnitudes[s] >= d->audio_channels ||
                m.angles[s] >= d->audio_channels) {
                rc = LWB_ERR_BAD_FORMAT;
                break;
            }
            dm.mag[s] = m.magnitudes[s];
            dm.ang[s] = m.angles[s];
        }
        for (int c = 0; c < d->audio_channels && rc == LWB_OK; c++) {
            if (m.mux[c] >= m.submaps || m.submap_floors[m.mux[c]] >= d->n_floors) {
                rc = LWB_ERR_BAD_FORMAT;      // header.rs:1023-1026, 1043-1047
                break;
            }
            dm.floor_of_channel[c] = m.submap_floors[m.mux[c]];
            if (d->audio_channels <= 8) dm.sub_ch[m.mux[c]][dm.sub_nch[m.mux[c]]++] = (uint8_t)c;
        }
    }
    for (uint32_t i = 0; i < d->n_modes && rc == LWB_OK; i++) {
        if (d->modes[i].mapping >= d->n_mappings) { rc = LWB_ERR_BAD_FORMAT; break; }   // header.rs:1067-1072
        su->host.mode_blockflag[i] = d->modes[i].blockflag ? 1 : 0;
        su->host.mode_mapping[i] = d->modes[i].mapping;
    }
    // LWB_ENTRY_VQ: codebook value tables and residue partition sizes
    if (rc == LWB_OK && d->n_codebooks) {
        if (d->n_codebooks > 256 || !d->codebooks || d->n_residues > (uint32_t)kMaxResidues || (d->n_residues && !d->residues)) {
            rc = LWB_ERR_INVALID;
        } else {
            std::vector<DevBook> books(d->n_codebooks);
            for (uint32_t i = 0; i < d->n_codebooks && rc == LWB_OK; i++) {
                const lwb_codebook_desc &cb = d->codebooks[i];
                books[i].vq = nullptr;
                books[i].entries = cb.entries;
                books[i].dims = cb.dimensions;
                books[i].pad = 0;
                if (cb.vq && cb.entries && cb.dimensions) rc = upload(su, cb.vq, (size_t)cb.entries * cb.dimensions, &books[i].vq);
            }
            if (rc == LWB_OK) rc = upload(su, books.data(), books.size(), &su->host.books);
            // (the uploads read the caller's tables: done before we return, see the synchronise below)
            if (rc == LWB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = LWB_ERR_CUDA;
            su->host.n_books = d->n_codebooks;
            su->host.n_residues = d->n_residues;
            for (uint32_t i = 0; i < d->n_residues; i++) su->host.res_psize[i] = d->residues[i].partition_size;
        }
    }
    if (rc == LWB_OK) rc = upload(su, floors.data(), floors.size(), &su->host.floors);
    if (rc == LWB_OK) rc = upload(su, su->mappings.data(), su->mappings.size(), &su->host.mappings);
    su->host.channels = d->audio_channels;
    su->host.bs0 = d->blocksize_0;
    su->host.bs1 = d->blocksize_1;
    su->host.n_floors = (uint8_t)d->n_floors;
    if (rc == LWB_OK) {
        const DevSetup *dp = nullptr;
        rc = upload(su, &su->host, 1, &dp);
        su->d_setup = const_cast<DevSetup *>(dp);
    }
    if (rc == LWB_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = LWB_ERR_CUDA;
    if (rc != LWB_OK) {
        lwb_setup_destroy(su);
        if (ctx->err.empty() || rc != LWB_ERR_CUDA) ctx->err = "setup: rejected (see header.rs validation rules)";
        return rc;
    }
    *out = su;
    return LWB_OK;
}

// ---------------------------------------------------------------------------------------------
// stream state
// ---------------------------------------------------------------------------------------------
static size_t state_stride(const lwb_setup *su) { return (size_t)1 << (su->bs1 - 1); }

extern "C" int lwb_stream_open(lwb_ctx *ctx, const lwb_setup *su, lwb_stream **out)
{
    if (!ctx || !su || !out || su->ctx != ctx) return LWB_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    lwb_stream *s = new (std::nothrow) lwb_stream();
    if (!s) return LWB_ERR_BUFFER;
    s->ctx = ctx;
    s->setup = su;
    cudaError_t e = cudaMalloc((void **)&s->d_state, su->channels * state_stride(su) * sizeof(float));
    if (e != cudaSuccess) {
        delete s;
        return fail(ctx, LWB_ERR_CUDA, "stream_open: cudaMalloc", e);
    }
    *out = s;
    return LWB_OK;
}

extern "C" void lwb_stream_destroy(lwb_stream *s)
{
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    cudaFree(s->d_state);
    delete s;
}

extern "C" int lwb_stream_reset(lwb_stream *s)
{
    if (!s) return LWB_ERR_INVALID;
    set_stream_state(s, false, 0);
    return LWB_OK;
}
extern "C" int lwb_stream_is_empty(const lwb_stream *s) { return (!s || !s->has) ? 1 : 0; }
extern "C" uint32_t lwb_stream_state_len(const lwb_stream *s) { return (s && s->has) ? s->plen : 0; }

extern "C" int lwb_stream_clone(const lwb_stream *s, lwb_stream **out)
{
    if (!s || !out) return LWB_ERR_INVALID;
    int rc = lwb_stream_open(s->ctx, s->setup, out);
    if (rc) return rc;
    (*out)->has = s->has;
    (*out)->plen = s->plen;
    lwb_ctx *ctx = s->ctx;
    CU(ctx, cudaMemcpyAsync((*out)->d_state, s->d_state,
                            s->setup->channels * state_stride(s->setup) * sizeof(float),
                            cudaMemcpyDeviceToDevice, ctx->stream));
    return LWB_OK;
}

extern "C" int lwb_stream_export_state(lwb_stream *s, float *out)
{
    if (!s || !out) return LWB_ERR_INVALID;
    if (!s->has) return LWB_OK;
    lwb_ctx *ctx = s->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpy2DAsync(out, s->plen * sizeof(float), s->d_state, state_stride(s->setup) * sizeof(float),
                              s->plen * sizeof(float), s->setup->channels, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return LWB_OK;
}

extern "C" int lwb_stream_import_state(lwb_stream *s, const float *data, uint32_t len)
{
    if (!s || (!data && len)) return LWB_ERR_INVALID;
    if (len > state_stride(s->setup)) return LWB_ERR_BUFFER;
    lwb_ctx *ctx = s->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (len) {
        CU(ctx, cudaMemcpy2DAsync(s->d_state, state_stride(s->setup) * sizeof(float), data, len * sizeof(float),
                                  len * sizeof(float), s->setup->channels, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    s->ctx->state_gen++;           // contents changed even if the shape did not
    s->has = true;
    s->plen = len;
    return LWB_OK;
}

extern "C" int lwb_decoded_sample_count(const lwb_setup *su, uint8_t mode, int prev_flag, int next_flag,
                                        uint32_t *n_samples)
{
    if (!su || !n_samples) return LWB_ERR_INVALID;
    Geom g;
    int rc = geometry(su, mode, prev_flag, next_flag, &g);
    if (rc) return rc;
    *n_samples = g.rs - g.ls;
    return LWB_OK;
}

#include "path_generic.cuh"
#include "path_long.cuh"
#include "path_chain.cuh"
#include "path_mixed.cuh"
#include "path_mid.cuh"

static int decode_chains_impl(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io, lwb_plan *prepared)
{
    if (!ctx || (!chains && n_chains) || !io) return LWB_ERR_INVALID;
    if (io->entry != LWB_ENTRY_SPECTRUM && io->entry != LWB_ENTRY_RESIDUE && io->entry != LWB_ENTRY_VQ) return fail(ctx, LWB_ERR_INVALID, "bad entry");
    if (io->memory != LWB_MEM_HOST && io->memory != LWB_MEM_DEVICE) return fail(ctx, LWB_ERR_INVALID, "bad memory space");
    if (io->out_format < 0 || io->out_format > LWB_OUT_I16_INTERLEAVED) return fail(ctx, LWB_ERR_INVALID, "bad out_format");
    if (n_chains == 0) return LWB_OK;
    if ((!io->coeffs && io->entry != LWB_ENTRY_VQ) || !io->pcm) return fail(ctx, LWB_ERR_INVALID, "null arena");
    if (io->entry == LWB_ENTRY_VQ && (!io->vq_runs || !io->vq_run_offsets || !io->vq_entries || !io->vq_entry_offsets || !io->floor_kind))
        return fail(ctx, LWB_ERR_INVALID, "VQ entry needs vq_runs, vq_entries, their offsets and floor_kind");
    CU(ctx, cudaSetDevice(ctx->device));
    const uint64_t epoch = ++ctx->epoch;      // per context: concurrent calls on different contexts share nothing
    {
        bool handled = false;
        const char *fg = getenv("LWB_FORCE_GENERIC");
        const bool no_fused = fg && std::strcmp(fg, "2") == 0;
        int rc0 = no_fused ? LWB_OK : try_long(ctx, chains, n_chains, io, epoch, &handled, nullptr, 0, prepared);
        if (rc0 || handled) return rc0;
        // residue-entry batches of uniform long blocks go front stages + fused kernel; everything else that fits
        // goes to the segmented path or the chain kernel
        if (!no_fused && !fg) {
            rc0 = try_long_residue(ctx, chains, n_chains, io, epoch, &handled, prepared);
            if (rc0 || handled) return rc0;
        }
        {
            if (!no_fused) {
                rc0 = try_mid(ctx, chains, n_chains, io, epoch, &handled, prepared);
                if (rc0 || handled) return rc0;
                rc0 = try_mixed(ctx, chains, n_chains, io, epoch, &handled, prepared);
                if (rc0 || handled) return rc0;
            }
            rc0 = try_chain(ctx, chains, n_chains, io, epoch, &handled, prepared);
            if (rc0 || handled) return rc0;
        }
    }
    const bool vq = io->entry == LWB_ENTRY_VQ;
    const bool residue = io->entry != LWB_ENTRY_SPECTRUM;
    const bool planar = is_planar(io->out_format);
    std::vector<PlanChain> plan(n_chains);
    uint64_t c_lo = ~0ull, c_hi = 0, o_lo = ~0ull, o_hi = 0, r_lo = ~0ull, r_hi = 0;
    int uniform_c = -1;
    bool need_dense = false;
    for (size_t i = 0; i < n_chains; i++) {
        lwb_chain *c = &chains[i];
        if (!c->stream || c->stream->ctx != ctx || (c->n_packets && !c->mode_numbers))
            return fail(ctx, LWB_ERR_INVALID, "chain: bad stream or mode list");
        if (c->stream->busy_epoch == epoch) return fail(ctx, LWB_ERR_INVALID, "a stream appears in two chains of one batch");
        c->stream->busy_epoch = epoch;
        const int C = c->stream->setup->channels;
        if (residue) {
            if (uniform_c < 0) uniform_c = C;
            if (uniform_c != C) return fail(ctx, LWB_ERR_INVALID, "residue batches need one channel count");
            if (!io->floor_kind) return fail(ctx, LWB_ERR_INVALID, "residue entry needs floor_kind");
        }
        plan_chain(c, &plan[i]);
        PlanChain &pc = plan[i];
        if (pc.pk.empty()) continue;
        const PlanPacket &last = pc.pk.back();
        c_lo = std::min(c_lo, c->coeff_offset);
        c_hi = std::max(c_hi, last.coeff_off + (uint64_t)C * (last.g.n >> 1));
        const uint64_t ext = planar ? (uint64_t)(C - 1) * c->out_stride + c->n_samples : (uint64_t)c->n_samples * C;
        if (planar && c->out_stride < c->n_samples) return fail(ctx, LWB_ERR_BUFFER, "chain: out_stride smaller than the samples produced");
        o_lo = std::min(o_lo, c->out_offset);
        o_hi = std::max(o_hi, c->out_offset + ext);
        if (residue) {
            r_lo = std::min(r_lo, c->packet_index);
            r_hi = std::max<uint64_t>(r_hi, c->packet_index + pc.pk.size());
            int krc = scan_floor_kinds(ctx, io, c->packet_index * C, (c->packet_index + pc.pk.size()) * C, &need_dense);
            if (krc) return krc;
        }
    }
    if (need_dense && !io->dense_floor) return fail(ctx, LWB_ERR_INVALID, "dense_floor missing");
    int rc = LWB_OK;
    if (c_hi > c_lo) {
        DevArenas ar = DevArenas();
        const size_t esz = elem_size(io->out_format);
        if (io->memory == LWB_MEM_HOST) {
            // stage: H2D of the used coefficient range, D2H of the used pcm range
            if (o_hi > o_lo && (rc = ensure(ctx, ctx->pcm, (o_hi - o_lo) * esz))) return rc;
            if (!vq) {
                if ((rc = ensure(ctx, ctx->coeffs, (c_hi - c_lo) * sizeof(float)))) return rc;
                CU(ctx, cudaMemcpyAsync(ctx->coeffs.p, io->coeffs + c_lo, (c_hi - c_lo) * sizeof(float),
                                        cudaMemcpyHostToDevice, ctx->stream));
                ar.coeffs = (const float *)ctx->coeffs.p;
            }
            ar.coeff_base = c_lo;
            if (need_dense) {
                if ((rc = ensure(ctx, ctx->dense, (c_hi - c_lo) * sizeof(float)))) return rc;
                CU(ctx, cudaMemcpyAsync(ctx->dense.p, io->dense_floor + c_lo, (c_hi - c_lo) * sizeof(float),
                                        cudaMemcpyHostToDevice, ctx->stream));
                ar.dense = (const float *)ctx->dense.p;
            }
            ar.pcm = ctx->pcm.p;
            ar.pcm_base = o_lo;
        } else {
            ar.coeffs = vq ? nullptr : io->coeffs;
            ar.dense = io->dense_floor;
            ar.pcm = io->pcm;
        }
        if ((rc = stage_vq_arrays(ctx, io, r_lo, r_hi, ctx->stream, &ar.vq))) return rc;
        if (residue) {
            // absolute packet rows address the (biased) device views: kinds_row0 stays 0
            if ((rc = stage_floor_arrays(ctx, io, r_lo, r_hi, (unsigned)uniform_c, ctx->stream, &ar.kinds, &ar.ys))) return rc;
            ar.kinds_row0 = 0;
        }
        if (residue && plan_is_long(plan, io)) {
            // residue entry, uniform long blocks: k_prologue forms the spectrum on the device, the fused
            // kernel does the rest (one extra spectrum round trip compared with the spectrum entry)
            if ((rc = run_prologue_all(ctx, plan, ar, (size_t)(c_hi - c_lo)))) return rc;
            bool handled = false;
            rc = try_long(ctx, chains, n_chains, io, epoch, &handled, (const float *)ctx->spec.p, ar.coeff_base);
            if (rc) return rc;
            if (handled) return LWB_OK;            // try_long has committed results and stream states
        }
        rc = run_generic(ctx, plan, io, ar);
        if (rc) return rc;
        if (io->memory == LWB_MEM_HOST) {
            if (o_hi > o_lo)
                CU(ctx, cudaMemcpyAsync((char *)io->pcm + o_lo * esz, ctx->pcm.p, (o_hi - o_lo) * esz,
                                        cudaMemcpyDeviceToHost, ctx->stream));
            CU(ctx, cudaStreamSynchronize(ctx->stream));
        }
    }
    // commit the host-side view of every stream's state
    for (auto &pc : plan) {
        lwb_stream *s = pc.c->stream;
        if (!pc.pk.empty() || pc.clear_after) set_stream_state(s, pc.end_has, pc.end_plen);
    }
    return LWB_OK;
}

extern "C" int lwb_decode_chains(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io)
{
    return decode_chains_impl(ctx, chains, n_chains, io, nullptr);
}

// ---------------------------------------------------------------------------------------------
// prepared batches
// ---------------------------------------------------------------------------------------------
extern "C" int lwb_plan_create(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io, lwb_plan **out)
{
    if (!ctx || !out || (!chains && n_chains) || !io) return LWB_ERR_INVALID;
    lwb_plan *p = new (std::nothrow) lwb_plan();
    if (!p) return LWB_ERR_BUFFER;
    p->ctx = ctx;
    p->chains = chains;
    p->n_chains = n_chains;
    p->io = *io;
    *out = p;
    return LWB_OK;
}

extern "C" void lwb_plan_destroy(lwb_plan *p)
{
    if (!p) return;
    if (p->runs.p || p->mix.p || p->pro.p) {
        cudaSetDevice(p->ctx->device);
        cudaStreamSynchronize(p->ctx->stream);
        if (p->runs.p) cudaFree(p->runs.p);
        if (p->mix.p) cudaFree(p->mix.p);
        if (p->pro.p) cudaFree(p->pro.p);
    }
    delete p;
}

// Replays the captured front stages of a residue-entry plan (device-memory batches only: host-memory batches are
// never captured as a whole).  Host floor arrays change from step to step and are uploaded again; device floor
// arrays are read in place.
static int replay_front_stages(lwb_plan *p)
{
    lwb_ctx *ctx = p->ctx;
    const lwb_batch_io *io = &p->io;
    const uint8_t *d_kinds;
    const uint32_t *d_ys;
    int rc = stage_floor_arrays(ctx, io, p->pro_r_lo, p->pro_r_hi, p->pro_C, ctx->stream, &d_kinds, &d_ys);
    if (rc) return rc;
    VqView vqv;
    if ((rc = stage_vq_arrays(ctx, io, p->pro_r_lo, p->pro_r_hi, ctx->stream, &vqv))) return rc;
    return launch_prologue(ctx, (const DevPacket *)p->pro.p, p->n_pro, p->pro_C, p->pro_fast, p->pro_smem_old, kLongN2,
                           io->entry == LWB_ENTRY_VQ ? nullptr : io->coeffs, io->dense_floor, d_kinds, d_ys, (float *)ctx->spec.p - p->pro_c_lo, vqv);
}

extern "C" int lwb_plan_execute(lwb_plan *p)
{
    if (!p) return LWB_ERR_INVALID;
    lwb_ctx *ctx = p->ctx;
    if (p->captured && p->gen == ctx->state_gen && !getenv("LWB_FORCE_GENERIC")) {
        // steady state: nothing about the batch or the stream states has changed shape since the
        // descriptors were built -- the per-chain results in the caller's array are still right,
        // the stream states stay (has, 1024): just launch.
        CU(ctx, cudaSetDevice(ctx->device));
        if (p->pro_captured) {             // residue entry: the front stages write ctx->spec, which the captured runs read
            int prc = replay_front_stages(p);
            if (prc) return prc;
        }
        constexpr uint32_t kTicketPool = 1024;
        if (ctx->ticket_next % kTicketPool == 0)
            CU(ctx, cudaMemsetAsync(ctx->ticket.p, 0, kTicketPool * sizeof(unsigned int), ctx->stream));
        unsigned int *ticket = (unsigned int *)ctx->ticket.p + (ctx->ticket_next++ % kTicketPool);
        if (long_launch(ctx->stream, (const LongRun *)p->runs.p, p->n_groups, p->pack, ticket, ctx->sm_count, p->i16, nullptr, 0, p->step))
            return fail(ctx, LWB_ERR_CUDA, "long kernel launch", cudaGetLastError());
        ctx->launches++;
        ctx->long_launches++;
        return LWB_OK;
    }
    if (p->mixed_captured && p->gen == ctx->state_gen && !getenv("LWB_FORCE_GENERIC")) {
        CU(ctx, cudaSetDevice(ctx->device));
        if (p->mix_pro) {                  // residue entry: front stages over every packet, then the rounds on ctx->spec
            const lwb_batch_io *io = &p->io;
            const uint8_t *d_kinds;
            const uint32_t *d_ys;
            int prc = stage_floor_arrays(ctx, io, p->mix_pro_r_lo, p->mix_pro_r_hi, p->mix_pro_C, ctx->stream, &d_kinds, &d_ys);
            if (prc) return prc;
            VqView vqv;
            if ((prc = stage_vq_arrays(ctx, io, p->mix_pro_r_lo, p->mix_pro_r_hi, ctx->stream, &vqv))) return prc;
            prc = launch_prologue(ctx, p->mix_pro_pk, p->mix_pro_n, p->mix_pro_C, p->mix_pro_fast, p->mix_pro_smem_old, p->mix_pro_n2max,
                                  io->entry == LWB_ENTRY_VQ ? nullptr : io->coeffs, p->mix_pro_dense ? io->dense_floor : nullptr, d_kinds, d_ys,
                                  (float *)ctx->spec.p - p->mix_pro_c_lo, vqv);
            if (prc) return prc;
        }
        return mixed_launch_rounds(ctx, p->mix_launch, p->mix_rounds);
    }
    return decode_chains_impl(ctx, p->chains, p->n_chains, &p->io, p);
}

// ---------------------------------------------------------------------------------------------
// one packet
// ---------------------------------------------------------------------------------------------
static int one_packet(lwb_stream *s, int entry, uint8_t mode, int prev_flag, int next_flag, const float *coeffs,
                      const lwb_packet *pkt, int out_format, void *out, size_t cap, size_t *n_samples)
{
    if (!s || !coeffs || !out || !n_samples) return LWB_ERR_INVALID;
    *n_samples = 0;
    Geom g;
    int rc = geometry(s->setup, mode, prev_flag, next_flag, &g);
    if (rc) return rc;
    const size_t produce = s->has ? g.rs - g.ls : 0;
    if (produce > cap) return LWB_ERR_BUFFER;          // checked before anything is consumed
    uint8_t m = mode, pf = (uint8_t)(prev_flag != 0), nf = (uint8_t)(next_flag != 0);
    lwb_chain c;
    std::memset(&c, 0, sizeof(c));
    c.stream = s;
    c.n_packets = 1;
    c.mode_numbers = &m;
    c.prev_window_flags = &pf;
    c.next_window_flags = &nf;
    c.out_stride = cap;
    lwb_batch_io io;
    std::memset(&io, 0, sizeof(io));
    io.entry = entry;
    io.memory = LWB_MEM_HOST;
    io.coeffs = coeffs;
    if (pkt) {
        io.dense_floor = pkt->dense_floor;
        io.floor_kind = pkt->floor_kind;
        io.floor1_y = pkt->floor1_y;
    }
    io.out_format = out_format;
    io.pcm = out;
    rc = lwb_decode_chains(s->ctx, &c, 1, &io);
    if (rc) return rc;
    if (c.status) return c.status;
    *n_samples = c.n_samples;
    return LWB_OK;
}

extern "C" int lwb_decode_packet(lwb_stream *s, const lwb_packet *pkt, int out_format, void *out, size_t cap,
                                 size_t *n_samples)
{
    if (!pkt || !pkt->floor_kind || !pkt->residue) return LWB_ERR_INVALID;
    return one_packet(s, LWB_ENTRY_RESIDUE, pkt->mode_number, pkt->prev_window_flag, pkt->next_window_flag,
                      pkt->residue, pkt, out_format, out, cap, n_samples);
}

extern "C" int lwb_decode_spectrum(lwb_stream *s, uint8_t mode, int prev_flag, int next_flag, const float *spectrum,
                                   int out_format, void *out, size_t cap, size_t *n_samples)
{
    return one_packet(s, LWB_ENTRY_SPECTRUM, mode, prev_flag, next_flag, spectrum, nullptr, out_format, out, cap,
                      n_samples);
}

// ---------------------------------------------------------------------------------------------
// debug taps (lib.rs:56-94): intermediates of one packet, state untouched
// ---------------------------------------------------------------------------------------------
extern "C" int lwb_debug_packet_taps(lwb_stream *s, const lwb_packet *pkt, float *post_inverse, float *pre_mdct,
                                     float *post_mdct)
{
    if (!s || !pkt || !pkt->floor_kind || !pkt->residue) return LWB_ERR_INVALID;
    lwb_ctx *ctx = s->ctx;
    const lwb_setup *su = s->setup;
    Geom g;
    int rc = geometry(su, pkt->mode_number, pkt->prev_window_flag, pkt->next_window_flag, &g);
    if (rc) return rc;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t C = su->channels, n2 = g.n >> 1;
    bool need_dense = false, need_y = false;
    for (size_t c = 0; c < C; c++) {
        if (pkt->floor_kind[c] > LWB_FLOOR_DENSE) return LWB_ERR_INVALID;
        need_dense |= pkt->floor_kind[c] == LWB_FLOOR_DENSE;
        need_y |= pkt->floor_kind[c] == LWB_FLOOR_ONE;
    }
    if ((need_dense && !pkt->dense_floor) || (need_y && !pkt->floor1_y)) return LWB_ERR_INVALID;
    if ((rc = ensure(ctx, ctx->coeffs, C * n2 * 4)) || (rc = ensure(ctx, ctx->spec, C * n2 * 4)) ||
        (rc = ensure(ctx, ctx->x, C * g.n * 4)) || (rc = ensure(ctx, ctx->kinds, C)) ||
        (rc = ensure(ctx, ctx->ys, C * LWB_MAX_POSTS * 4)) || (rc = ensure(ctx, ctx->dense, C * n2 * 4)) ||
        (rc = ensure(ctx, ctx->desc, sizeof(DevPacket))) || (rc = ensure_pinned(ctx, sizeof(DevPacket))))
        return rc;
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    DevPacket *d = (DevPacket *)ctx->h_desc;
    std::memset(d, 0, sizeof(*d));
    d->setup = su->d_setup;
    d->state = s->d_state;
    d->prev_packet = -1;
    d->state_stride = (uint32_t)state_stride(su);
    d->n = (uint16_t)g.n;
    d->ls = (uint16_t)g.ls; d->rs = (uint16_t)g.rs; d->re = (uint16_t)g.re;
    d->blockflag = g.blockflag; d->mapping = g.mapping; d->slope_sel = g.slope_sel;
    d->channels = (uint8_t)C;
    cudaStream_t st = ctx->stream;
    CU(ctx, cudaMemcpyAsync(ctx->desc.p, d, sizeof(*d), cudaMemcpyHostToDevice, st));
    CU(ctx, cudaMemcpyAsync(ctx->coeffs.p, pkt->residue, C * n2 * 4, cudaMemcpyHostToDevice, st));
    CU(ctx, cudaMemcpyAsync(ctx->kinds.p, pkt->floor_kind, C, cudaMemcpyHostToDevice, st));
    if (need_y) CU(ctx, cudaMemcpyAsync(ctx->ys.p, pkt->floor1_y, C * LWB_MAX_POSTS * 4, cudaMemcpyHostToDevice, st));
    if (need_dense) CU(ctx, cudaMemcpyAsync(ctx->dense.p, pkt->dense_floor, C * n2 * 4, cudaMemcpyHostToDevice, st));
    const DevPacket *dp = (const DevPacket *)ctx->desc.p;
    if (post_inverse) {
        // audio.rs:1004 tap: coupling only -- run the prologue with every floor "dense = 1.0"?  No:
        // the tap is taken by running the prologue on a copy with all floors unused replaced by a
        // unit curve, so that floor x residue leaves the decoupled residue unchanged.
        std::vector<float> ones(C * n2, 1.0f);
        std::vector<uint8_t> kd(C, LWB_FLOOR_DENSE);
        void *tmp_dense = nullptr, *tmp_kinds = nullptr;
        CU(ctx, cudaMalloc(&tmp_dense, C * n2 * 4));
        CU(ctx, cudaMalloc(&tmp_kinds, C));
        CU(ctx, cudaMemcpyAsync(tmp_dense, ones.data(), C * n2 * 4, cudaMemcpyHostToDevice, st));
        CU(ctx, cudaMemcpyAsync(tmp_kinds, kd.data(), C, cudaMemcpyHostToDevice, st));
        rc = launch(ctx, k_prologue, dim3(1), dim3(kPrologueThreads), prologue_smem(su->channels, su->bs1), dp, (const float *)ctx->coeffs.p,
                    (const float *)tmp_dense, (const uint8_t *)tmp_kinds, (const uint32_t *)ctx->ys.p,
                    (float *)ctx->spec.p);
        if (!rc) {
            cudaError_t e = cudaMemcpyAsync(post_inverse, ctx->spec.p, C * n2 * 4, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) rc = fail(ctx, LWB_ERR_CUDA, "tap copy", e);
        }
        cudaFree(tmp_dense);
        cudaFree(tmp_kinds);
        if (rc) return rc;
    }
    if ((rc = launch(ctx, k_prologue, dim3(1), dim3(kPrologueThreads), prologue_smem(su->channels, su->bs1), dp, (const float *)ctx->coeffs.p,
                     (const float *)ctx->dense.p, (const uint8_t *)ctx->kinds.p, (const uint32_t *)ctx->ys.p,
                     (float *)ctx->spec.p)))
        return rc;
    if (pre_mdct) CU(ctx, cudaMemcpyAsync(pre_mdct, ctx->spec.p, C * n2 * 4, cudaMemcpyDeviceToHost, st));
    if (post_mdct) {
        if ((rc = launch(ctx, k_imdct, dim3(1, (unsigned)C), dim3(kImdctThreads), g.n * sizeof(float), dp,
                         (const float *)ctx->spec.p, (float *)ctx->x.p)))
            return rc;
        CU(ctx, cudaMemcpyAsync(post_mdct, ctx->x.p, C * g.n * 4, cudaMemcpyDeviceToHost, st));
    }
    CU(ctx, cudaStreamSynchronize(st));
    return LWB_OK;
}

