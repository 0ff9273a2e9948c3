/*
 * lewton_b200.h -- C ABI of the B200-native Vorbis packet-synthesis back-end.
 *
 * What it replaces (RustAudio/lewton @ bb2955b): the dense back half of
 *   audio::read_audio_packet_generic            src/audio.rs:988-1157
 * i.e. inverse channel coupling (:991-1002), floor-1 curve synthesis
 * (:391-555) and floor x residue (:1006-1039), imdct::inverse_mdct
 * (src/imdct.rs:291-659), window / overlap-add / PreviousWindowRight
 * (:1056-1154) and Samples::from_floats (src/samples.rs:20-103).  The bit-serial
 * front half (:921-986: mode bits, floor_decode, residue_packet_decode) stays in
 * Rust on the host and hands its dense results across this boundary.
 *
 * Style follows the crate's own C API (src/capi.rs:78-147): opaque pointers,
 * int status, out-parameters, explicit *_destroy.  Nothing unwinds across the
 * boundary.  There is NO CPU fallback: every entry point that computes fails
 * with LWB_ERR_NO_DEVICE / LWB_ERR_CUDA when no sm_100 device is usable.
 *
 * Threading: a ctx is bound to one CUDA device and is not thread-safe (the
 * reference is single-threaded and &mut-exclusive per stream); use one ctx per
 * host thread / per GPU.  Streams of one ctx are independent; packets of one
 * stream must be submitted in order (overlap-add dependency).
 *
 * All arithmetic is IEEE binary32, round-to-nearest, never contracted, in the
 * reference's operation order: f32 PCM is bit-identical to lewton's own output
 * (up to the sign of zero / NaN payload), i16 PCM is bit-identical.
 */
#ifndef LEWTON_B200_H
#define LEWTON_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LWB_ABI_VERSION 3          /* 2: lwb_batch_io::floor_memory, lwb_bind_host_to_device; 3: LWB_ENTRY_VQ */
#define LWB_MAX_POSTS 65          /* header.rs:873 floor1_values <= 65 */
#define LWB_MAX_CHANNELS 255      /* audio_channels is a u8, header.rs:190 */
#define LWB_MAX_COUPLING 256      /* header.rs:998-1001 coupling steps = read_u8 + 1 */
#define LWB_MAX_SUBMAPS 16        /* header.rs:994-997 submaps = read_u4 + 1 */
#define LWB_MAX_MODES 64          /* header.rs:1134 mode count = read_u6 + 1 */

/* status codes (0 = ok), cf. audio::AudioReadError (audio.rs:26-41) */
enum {
    LWB_OK = 0,
    LWB_ERR_BAD_FORMAT = 1,   /* AudioReadError::AudioBadFormat (mode index, OLA guard :1107-1111) */
    LWB_ERR_BUFFER = 2,       /* AudioReadError::BufferNotAddressable / output capacity too small */
    LWB_ERR_MISMATCH = 3,     /* where the reference panics: channel-count mismatch (:1086), mag==ang (:783) */
    LWB_ERR_INVALID = 4,      /* NULL / out-of-range argument */
    LWB_ERR_CUDA = 5,         /* a CUDA call failed; see lwb_last_error */
    LWB_ERR_NO_DEVICE = 6     /* no usable sm_100 device: there is no CPU fallback */
};

typedef struct lwb_ctx lwb_ctx;        /* one per GPU: stream, staging, launch state           */
typedef struct lwb_setup lwb_setup;    /* what IdentHeader + SetupHeader give the synthesis half */
typedef struct lwb_stream lwb_stream;  /* PreviousWindowRight (audio.rs:847-861), device-resident */

/* ---- library / context ------------------------------------------------------------------ */
int lwb_abi_version(void);
/* number of CUDA devices visible (0 on a CPU-only host; never fails) */
int lwb_device_count(void);
int lwb_ctx_create(int device_ordinal, lwb_ctx **out);
void lwb_ctx_destroy(lwb_ctx *ctx);
/* block until everything submitted on this ctx has finished */
int lwb_ctx_synchronize(lwb_ctx *ctx);
/* text of the last failure on this ctx (never NULL) */
const char *lwb_last_error(const lwb_ctx *ctx);
/* the cudaStream_t all work of this ctx is launched on (for CUDA-event timing by a harness) */
void *lwb_ctx_cuda_stream(lwb_ctx *ctx);
/* kernels launched by this ctx since creation (bench.py's gpu_launches) */
uint64_t lwb_ctx_launch_count(const lwb_ctx *ctx);
/* of those, launches of the fused long-block kernels (k_long, k_long_s): tells the fused path from the chain kernel */
uint64_t lwb_ctx_long_launch_count(const lwb_ctx *ctx);
/* pinned host memory for the host-buffer entry points (optional; plain malloc'd memory works, slower) */
void *lwb_host_alloc(size_t bytes);
void lwb_host_free(void *p);
/* Multi-GPU hosts: bind the calling thread (and the threads it creates) to the CPUs of the NUMA node GPU
 * `device_ordinal` is attached to and prefer that node's memory, so that pinned buffers allocated afterwards
 * (lwb_host_alloc, staging) are local to the GPU's PCIe root.  Call once per rank / per feeding thread before
 * allocating.  Returns the node, or -1 if unknown (nothing changed).  device_ordinal < 0 restores the default
 * memory policy (the CPU affinity is the caller's to restore).  No reference counterpart: lewton is CPU-only. */
int lwb_bind_host_to_device(int device_ordinal);
/* device memory helpers for the *_DEVICE memory space (harnesses without their own allocator) */
int lwb_device_alloc(lwb_ctx *ctx, size_t bytes, void **out);
void lwb_device_free(lwb_ctx *ctx, void *p);
int lwb_memcpy_h2d(lwb_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int lwb_memcpy_d2h(lwb_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);

/* ---- blocksize-derived tables: header_cached.rs:33-110 ----------------------------------- */
/* CachedBlocksizeDerived::from_blocksize, evaluated on the host with libm sinf/cosf in the
 * reference's f32 expression order.  a,b: n/2 floats; c: n/4; window: n/2; bitrev: n/8. */
int lwb_tables_generate(int blocksize_log2, float *a, float *b, float *c, float *window,
                        uint32_t *bitrev);

/* ---- setup: the header-derived constants the synthesis half reads ------------------------- */
typedef struct lwb_tables_ref {      /* IdentHeader.cached_bs_derived[i], header.rs:210           */
    const float *a, *b, *c;          /* TwiddleFactors, header_cached.rs:20-24                     */
    const float *window;             /* window_slope                                               */
    const uint32_t *bitrev;
} lwb_tables_ref;

enum { LWB_FLOOR_TYPE_ZERO = 0, LWB_FLOOR_TYPE_ONE = 1 };
typedef struct lwb_floor_desc {      /* header::Floor, header.rs:399-424                           */
    uint8_t floor_type;              /* type 0 curves are computed by the host and passed dense    */
    uint8_t floor1_multiplier;       /* 1..4                                                       */
    uint8_t floor1_values;           /* floor1_x_list.len(), 2..65                                 */
    uint8_t reserved;
    uint32_t floor1_x_list[LWB_MAX_POSTS];   /* unsorted, as parsed (header.rs:878-884)            */
} lwb_floor_desc;

typedef struct lwb_mapping_desc {    /* header::Mapping, header.rs:384-390                         */
    uint16_t coupling_steps;
    uint8_t submaps;
    uint8_t reserved;
    uint8_t magnitudes[LWB_MAX_COUPLING];
    uint8_t angles[LWB_MAX_COUPLING];
    uint8_t mux[LWB_MAX_CHANNELS + 1];       /* mapping_mux[channel] -> submap                     */
    uint8_t submap_floors[LWB_MAX_SUBMAPS];  /* submap -> floor index                              */
} lwb_mapping_desc;

typedef struct lwb_mode_desc {       /* header::ModeInfo, header.rs:393-396                        */
    uint8_t blockflag;
    uint8_t mapping;
} lwb_mode_desc;

/* Codebook value tables and residue shapes (only for LWB_ENTRY_VQ batches; leave the counts 0 otherwise). */
typedef struct lwb_codebook_desc {   /* header::Codebook, header.rs:360-368                            */
    uint16_t dimensions;             /* codebook_dimensions                                            */
    uint16_t reserved;
    uint32_t entries;                /* codebook_entries                                               */
    const float *vq;                 /* codebook_vq_lookup_vec: [entries][dimensions]; NULL = no value mapping */
} lwb_codebook_desc;
typedef struct lwb_residue_desc {    /* header::Residue, header.rs:370-379                             */
    uint8_t residue_type;            /* 0, 1, 2                                                        */
    uint8_t reserved[3];
    uint32_t partition_size;         /* residue_partition_size                                         */
} lwb_residue_desc;

typedef struct lwb_setup_desc {
    uint8_t audio_channels;          /* IdentHeader.audio_channels                                 */
    uint8_t blocksize_0, blocksize_1;/* log2, 6..13, blocksize_0 <= blocksize_1 (header.rs:239-243)    */
    uint8_t reserved;
    /* optional: the crate's own tables (so results cannot depend on the libm behind them);
     * a NULL `a` means "generate with lwb_tables_generate" */
    lwb_tables_ref tables[2];
    uint32_t n_floors;
    const lwb_floor_desc *floors;
    uint32_t n_mappings;
    const lwb_mapping_desc *mappings;
    uint32_t n_modes;
    const lwb_mode_desc *modes;
    /* LWB_ENTRY_VQ only (ABI 3; zero / NULL otherwise) */
    uint32_t n_codebooks;
    const lwb_codebook_desc *codebooks;
    uint32_t n_residues;
    const lwb_residue_desc *residues;
} lwb_setup_desc;

int lwb_setup_create(lwb_ctx *ctx, const lwb_setup_desc *desc, lwb_setup **out);
void lwb_setup_destroy(lwb_setup *setup);

/* ---- stream state: PreviousWindowRight, audio.rs:847-861 ---------------------------------- */
int lwb_stream_open(lwb_ctx *ctx, const lwb_setup *setup, lwb_stream **out);
void lwb_stream_destroy(lwb_stream *s);
/* PreviousWindowRight::new(): the next packet yields 0 samples (audio.rs:1140-1151) */
int lwb_stream_reset(lwb_stream *s);
/* PreviousWindowRight::is_empty() */
int lwb_stream_is_empty(const lwb_stream *s);
/* #[derive(Clone)]: an independent copy of the state */
int lwb_stream_clone(const lwb_stream *s, lwb_stream **out);
/* debug / checkpoint: per-channel length of the saved right half (0 if empty), and its data */
uint32_t lwb_stream_state_len(const lwb_stream *s);
int lwb_stream_export_state(lwb_stream *s, float *out /* [channels][len] */);
int lwb_stream_import_state(lwb_stream *s, const float *data /* [channels][len] */, uint32_t len);

/* audio::get_decoded_sample_count (audio.rs:874-909) for an already-parsed packet header:
 * right_win_start - left_win_start; does not look at the stream state. */
int lwb_decoded_sample_count(const lwb_setup *setup, uint8_t mode_number, int prev_window_flag,
                             int next_window_flag, uint32_t *n_samples);

/* ---- one packet (mirrors read_audio_packet_generic's back half) --------------------------- */
enum { LWB_FLOOR_UNUSED = 0,   /* DecodedFloor::Unused  -> zero curve (audio.rs:1021-1024)        */
       LWB_FLOOR_ONE = 1,      /* DecodedFloor::TypeOne -> raw floor1_y from floor_one_decode      */
       LWB_FLOOR_DENSE = 2 };  /* DecodedFloor::TypeZero -> curve computed by the host (n/2 f32)   */

enum { LWB_OUT_F32_PLANAR = 0,        /* Vec<Vec<f32>>            samples.rs:20-40, 86-90          */
       LWB_OUT_I16_PLANAR = 1,        /* Vec<Vec<i16>>            samples.rs:92-103                */
       LWB_OUT_F32_INTERLEAVED = 2,   /* InterleavedSamples<f32>  samples.rs:43-79                 */
       LWB_OUT_I16_INTERLEAVED = 3 }; /* InterleavedSamples<i16>                                   */

typedef struct lwb_packet {
    uint8_t mode_number;             /* audio.rs:925                                               */
    uint8_t prev_window_flag;        /* audio.rs:935, long blocks only (ignored for short ones)    */
    uint8_t next_window_flag;
    uint8_t reserved;
    const uint8_t *floor_kind;       /* [channels] LWB_FLOOR_*                                     */
    const uint32_t *floor1_y;        /* [channels][LWB_MAX_POSTS] rows used where kind == ONE      */
    const float *dense_floor;        /* [channels][n/2], rows used where kind == DENSE, else NULL  */
    const float *residue;            /* [channels][n/2] after residue_packet_decode (audio.rs:986) */
} lwb_packet;

/* Synchronous convenience = submit + flush + fetch.  out: planar [channels][capacity] or
 * interleaved [capacity][channels]; *n_samples = samples per channel written (0 for the first
 * packet after a reset).  Host buffers. */
int lwb_decode_packet(lwb_stream *s, const lwb_packet *pkt, int out_format, void *out,
                      size_t capacity_per_channel, size_t *n_samples);
/* Entry at record_pre_mdct (audio.rs:1041): spectrum [channels][n/2] already floor x residue. */
int lwb_decode_spectrum(lwb_stream *s, uint8_t mode_number, int prev_window_flag,
                        int next_window_flag, const float *spectrum, int out_format, void *out,
                        size_t capacity_per_channel, size_t *n_samples);

/* ---- batches: many streams x consecutive packets in one submission ------------------------- */
enum { LWB_ENTRY_SPECTRUM = 0,   /* coeffs = floor x residue, enters at audio.rs:1041             */
       LWB_ENTRY_RESIDUE = 1,    /* coeffs = residue vectors, enters at audio.rs:988               */
       LWB_ENTRY_VQ = 2 };       /* no dense coefficients cross the boundary: the residue vectors are  *
                                  * accumulated on the device from the packets' VQ entry indices       *
                                  * (audio.rs:587-717); coeff_offset still lays out the (device-only)   *
                                  * coefficient arena.  Needs the setup's codebooks / residues, <= 8     *
                                  * channels, channels * n/2 <= 12288, VQ books of <= 65536 entries whose   *
                                  * dimension divides their residue's partition size.                     */
/* The VQ vectors of a packet's residue, in the order the entropy decoder produces them (SURVEY.md 8f rank 2), as RUNS:
 * one run = the consecutive vectors one residue_packet_read_partition call reads (audio.rs:587-618) -- same codebook,
 * same pass, positions in arithmetic progression -- plus one 16-bit codebook entry per vector in a side array.  The
 * f32 += order of the reference is kept on the device: per coefficient the contributions are added pass by pass
 * (audio.rs:595, :611); within a pass no two vectors of a packet touch the same coefficient. */
typedef struct lwb_vq_run {
    uint16_t pos;                    /* where vector 0 of the run lands (see kind)                          */
    uint16_t first;                  /* index of its entry in the packet's slice of vq_entries              */
    uint8_t book;                    /* codebook index                                                      */
    uint8_t pass_kind;               /* bits 0..2 pass (0..7), bits 3..4 kind:                                *
                                      *   0 contiguous in a channel vector (residue type 1): pos = channel * n/2 + bin,
                                      *     vector i at pos + i * dimensions
                                      *   1 strided (type 0, audio.rs:589-597): vector i at pos + i, its value j at
                                      *     + j * step, step = partition_size(aux) / dimensions
                                      *   2 interleaved (type 2, audio.rs:744-756): pos indexes the interleaved vector of
                                      *     submap `aux` (element t = channel t % ch, bin t / ch), vector i at pos + i * dimensions */
    uint8_t aux;                     /* kind 1: residue index; kind 2: submap index                          */
    uint8_t count;                   /* vectors in the run (a longer partition is split)                     */
} lwb_vq_run;
#define LWB_VQ_PASS_KIND(pass, kind) ((uint8_t)((pass) | ((kind) << 3)))
enum { LWB_MEM_HOST = 0, LWB_MEM_DEVICE = 1 };

/* One stream's run of consecutive packets.  Input arenas are chain-major: the chain's packets
 * follow each other, each packet as [channels][n/2 of that packet]. */
typedef struct lwb_chain {
    lwb_stream *stream;
    uint32_t n_packets;
    const uint8_t *mode_numbers;      /* [n_packets] (host memory)                                 */
    const uint8_t *prev_window_flags; /* [n_packets] or NULL = all 1                               */
    const uint8_t *next_window_flags; /* [n_packets] or NULL = all 1                               */
    uint64_t coeff_offset;            /* element offset of the chain's first packet in `coeffs`    */
    uint64_t packet_index;            /* index of the chain's first packet in per-packet arenas    */
    uint64_t out_offset;              /* element offset of the chain's PCM in `pcm`                 */
    uint64_t out_stride;              /* planar: elements between channel planes (>= total samples)*/
    /* results */
    uint32_t n_samples;               /* samples per channel produced by this chain                */
    uint32_t packets_done;            /* == n_packets unless status != 0                           */
    int32_t status;                   /* LWB_OK or the error of packet `packets_done`              */
} lwb_chain;

typedef struct lwb_batch_io {
    int entry;                        /* LWB_ENTRY_*                                               */
    int memory;                       /* LWB_MEM_*: where coeffs/dense_floor/pcm live              */
    const float *coeffs;              /* spectrum or residue arena                                 */
    const float *dense_floor;         /* same layout as coeffs, or NULL (LWB_ENTRY_RESIDUE)        */
    const uint8_t *floor_kind;        /* [total_packets][channels]   (LWB_ENTRY_RESIDUE), see floor_memory */
    const uint32_t *floor1_y;         /* [total_packets][channels][LWB_MAX_POSTS], see floor_memory */
    int out_format;                   /* LWB_OUT_*                                                 */
    void *pcm;                        /* output arena                                              */
    /* LWB_ENTRY_VQ: the runs / entries of packet row r (= chain.packet_index + k); all four arrays live where the    *
     * floor arrays live (floor_memory).                                                                            */
    const lwb_vq_run *vq_runs;
    const uint64_t *vq_run_offsets;   /* [total_packets + 1]: packet row r owns vq_runs[off[r] .. off[r + 1])          */
    const uint16_t *vq_entries;
    const uint64_t *vq_entry_offsets; /* [total_packets + 1]: ... and vq_entries[eoff[r] .. eoff[r + 1])            */
    int floor_memory;                 /* LWB_MEM_*: where floor_kind / floor1_y live (0 = host).   *
                                       * Device arrays are read in place (nothing is uploaded, and   *
                                       * nothing about them can be validated on the host: a kind    *
                                       * outside LWB_FLOOR_* acts as LWB_FLOOR_UNUSED); a decode     *
                                       * server whose entropy stage fills device-visible buffers     *
                                       * submits residue-entry batches without any per-step copy.   */
} lwb_batch_io;

/* All chains must use setups with the same channel count per chain's own stream; chains may
 * mix setups.  Returns LWB_OK when the batch ran (per-chain status holds format errors), or a
 * CUDA / argument error.  With LWB_MEM_HOST the call returns after the PCM has landed in `pcm`;
 * with LWB_MEM_DEVICE it returns after the launches are enqueued on lwb_ctx_cuda_stream(). */
int lwb_decode_chains(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io);

/* Prepared batches.  A decode server submits the same batch shape step after step (same streams,
 * same packets per stream, same arenas); planning it again each time costs more host time than
 * the GPU needs to run it.  lwb_plan_create captures the chain array, the io block and the
 * per-chain mode / flag arrays BY REFERENCE (they must stay valid and unchanged until
 * lwb_plan_destroy); lwb_plan_execute is then equivalent to lwb_decode_chains on that batch
 * -- same results, same stream-state updates, same per-chain outputs in the captured chain
 * array -- but reuses the device descriptors whenever no stream state has changed shape since they
 * were built (it re-plans by itself otherwise, e.g. on the first execution after a reset). */
typedef struct lwb_plan lwb_plan;
int lwb_plan_create(lwb_ctx *ctx, lwb_chain *chains, size_t n_chains, const lwb_batch_io *io, lwb_plan **out);
int lwb_plan_execute(lwb_plan *plan);
void lwb_plan_destroy(lwb_plan *plan);

/* Debug taps at the reference's record_* points (lib.rs:56-94; audio.rs:1004, 1041, 1054):
 * run one packet and return the intermediate vectors instead of PCM.  taps: any may be NULL.
 * post_inverse / pre_mdct: [channels][n/2]; post_mdct: [channels][n].  Does not touch the state. */
int lwb_debug_packet_taps(lwb_stream *s, const lwb_packet *pkt, float *post_inverse,
                          float *pre_mdct, float *post_mdct);

#ifdef __cplusplus
}
#endif
#endif /* LEWTON_B200_H */
