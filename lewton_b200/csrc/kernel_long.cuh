// kernel_long.cuh -- the hot path: fused IMDCT + window + overlap-add for runs of consecutive
// long blocks (n = 2048) of one channel.  One WARP owns one run: it walks the run's packets in
// order, keeps the previous block's right half in registers (the only inter-packet state,
// audio.rs:847-861), and emits 1024 f32 PCM samples per packet with fully coalesced stores.
// HBM traffic is the algorithmic minimum: 4 KB spectrum in (TMA bulk copy into shared memory,
// three tiles in flight per warp) + 4 KB PCM out per block.
//
// Arithmetic = the reference's butterfly network (imdct.rs:291-659), every add/sub/mul in the
// reference's operand order, unfused (bit parity); what is ours is the schedule:
//
//   complex view: z_c = U[2c+1] + i*U[2c], c in [0,512).  The step-3 stages are a radix-2 DIF FFT
//   over the 9 bits of c: step 2 flips bit 8, stage l flips bit 7-l, ld654 covers bits 2,1,0.
//   Each lane holds 16 complex values = 2 groups x 8 "slots"; the slot index carries 3 bits of c:
//     phase A: slot = bits 8,7,6   -> step 0 (pre-twiddle), step 2, stages 0 and 1, in registers
//     phase B: slot = bits 5,4,3   -> stages 2, 3, 4
//     phase C: slot = bits 2,1,0   -> ld654, bit-reverse (free: renaming), step 7, step 8, OLA
//   with two swizzled shared-memory transposes in between (conflict-free 32-bit accesses).
//   The two groups of a lane are chosen so that
//     * phase A: one float4 of spectrum feeds both groups (c and 511-c come from the same quad),
//     * phase C: the step-7 partner (c' <-> 511-c') of every value lives in the same lane,
//     * output index m = 64*rev3(slot) + lane (or 63-lane): every store is a full 128 B line.
//   Every operation is written on V = (group a, group b) pairs, which maps 1:1 onto Blackwell's
//   packed add/sub/mul.rn.f32x2 (SASS FADD2/FMUL2; IEEE RN per lane, so parity-safe) and halves
//   the FP issue slots of this issue-bound, non-FMA-able kernel.
//   Twiddles/window: a per-lane "pack" (built once per setup on the host from the uploaded
//   tables) is staged in shared memory per CTA; phases A/B keep theirs in registers across the
//   whole run, phase C reads its 48 pairs per block from the shared copy.
//
// The per-lane phase functions are plain inline functions of (lane, registers, twiddles): they
// also compile for the host, where tests/emu runs all 32 lanes sequentially against the oracle
// (test infrastructure only; the product never executes them on the CPU).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define LWB_HD __host__ __device__ __forceinline__
#else
#define LWB_HD inline
#endif

namespace lwb {

constexpr int kLongBs = 11;
constexpr int kLongN = 2048;
constexpr int kLongN2 = 1024;

// one run = consecutive packets of one channel of one stream
struct alignas(16) LongRun {      // 48 bytes: fetched by the kernel with one 1-D TMA copy
    const float *in;        // first packet's spectrum (1024 floats); next packet at +in_stride
    void *out;              // first emitted packet's PCM (f32 or i16 elements); next at +1024
    float *state;           // stream state row of this channel (1024 floats)
    uint32_t in_stride;
    uint32_t n_packets;     // including a primer packet if prime != 0
    uint8_t has_prev;       // 1: packet 0 overlaps with `state`;  0: packet 0 emits nothing
    uint8_t write_state;    // 1: store the last packet's right half to `state`
    uint8_t dummy;          // 1: filler partner of an unpaired run: transformed, never stored
    uint8_t first_short;    // 1: packet 0 follows a short block (previous_window_flag == 0, audio.rs:1059-1065);
                            // 2: the same, but the short block's kernel runs AFTER this one: packet 0 stores its
                            //    windowed left slope x[ls + i] w[i] (i < pl) to `state` instead of reading it, and
                            //    leaves the first pl PCM samples to that kernel (k_short's tail, which adds its half)
    uint8_t last_short;     // 1: the last packet precedes a short block (next_window_flag == 0, audio.rs:1067-1073)
    uint8_t pad[3];
    float *state_out;       // where write_state stores (nullptr: `state`)
};
static_assert(sizeof(LongRun) == 48, "LongRun is copied by TMA in 16-byte units");

struct V { float x, y; };    // (group a, group b)

#if defined(__CUDA_ARCH__)
#ifndef LWB_PACKED_F32X2
#define LWB_PACKED_F32X2 1
#endif
#if LWB_PACKED_F32X2
__device__ __forceinline__ unsigned long long v_bits(V a)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
    return r;
}
__device__ __forceinline__ V v_from(unsigned long long r)
{
    V a;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(r));
    return a;
}
__device__ __forceinline__ V vadd(V a, V b)
{
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(v_bits(a)), "l"(v_bits(b)));
    return v_from(r);
}
__device__ __forceinline__ V vsub(V a, V b)
{
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(v_bits(a)), "l"(v_bits(b)));
    return v_from(r);
}
__device__ __forceinline__ V vmul(V a, V b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(v_bits(a)), "l"(v_bits(b)));
    return v_from(r);
}
#else
__device__ __forceinline__ V vadd(V a, V b) { return V{__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)}; }
__device__ __forceinline__ V vsub(V a, V b) { return V{__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y)}; }
__device__ __forceinline__ V vmul(V a, V b) { return V{__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)}; }
#endif
// Add/sub whose operands are PRODUCTS.  ptxas (12.9) contracts mul.rn.f32x2 + add.rn.f32x2 into
// FFMA2 even with explicit .rn and -fmad=false (it also rewrites fma(a,b,-0) and fma(a,1,c) back
// to mul/add first), which would merge two of the reference's roundings into one.  Scalar
// add.rn.f32 is never contracted, so the product-consuming adds stay scalar (FADD) while all
// other adds and all multiplies are packed (FADD2 / FMUL2).
__device__ __forceinline__ V vadd_p(V a, V b) { return V{__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)}; }
__device__ __forceinline__ V vsub_p(V a, V b) { return V{__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y)}; }
// -(a) - b for products: the scalar FADD takes both negations as free operand modifiers
__device__ __forceinline__ V vnsub_p(V a, V b) { return V{__fsub_rn(-a.x, b.x), __fsub_rn(-a.y, b.y)}; }
#else
// host (pack builder is host code; the phase functions run here only inside tests/emu).
// Compiled with -ffp-contract=off: one rounding per operation, like the device path.
inline V vadd(V a, V b) { return V{a.x + b.x, a.y + b.y}; }
inline V vsub(V a, V b) { return V{a.x - b.x, a.y - b.y}; }
inline V vmul(V a, V b) { return V{a.x * b.x, a.y * b.y}; }
inline V vadd_p(V a, V b) { return vadd(a, b); }
inline V vsub_p(V a, V b) { return vsub(a, b); }
inline V vnsub_p(V a, V b) { return V{-a.x - b.x, -a.y - b.y}; }
#endif

// ---- pack layout: V slots per lane, stored slot-major [slot][lane] --------------------------
enum {
    P_S0W0 = 0, P_S0W1 = 8,            // step 0 pre-twiddle, per slot
    P_S2W0 = 16, P_S2W1 = 20,          // step 2, butterflies (slot j, j+4), j < 4
    P_L0W0 = 24, P_L0W1 = 26,          // stage 0: index = slot & 1
    P_L1W0 = 28, P_L1W1 = 29,          // stage 1
    P_A_END = 30,
    P_L2W0 = 30, P_L2W1 = 34,          // stage 2: index = slot & 3
    P_L3W0 = 38, P_L3W1 = 40,          // stage 3: index = slot & 1
    P_L4W0 = 42, P_L4W1 = 43,          // stage 4
    P_B_END = 44,
    P_A2 = 44,                         // A[n/8] (ld654)
    P_S7C0 = 45, P_S7C1 = 49,          // step 7, odd slots 1,3,5,7 -> index slot >> 1
    P_B0 = 53, P_B1 = 61,              // step 8 per slot
    P_WLO = 69, P_WHI = 77,            // window w[m], w[1023-m] per slot
    P_END = 85
};
constexpr int kLongPackFloats = P_END * 32 * 2;

LWB_HD int rev3(int j) { return ((j & 1) << 2) | (j & 2) | ((j >> 2) & 1); }
LWB_HD int rev6(int t) { return (rev3(t & 7) << 3) | rev3((t >> 3) & 7); }
LWB_HD int rev9(int c) { return (rev3(c & 7) << 6) | (rev3((c >> 3) & 7) << 3) | rev3((c >> 6) & 7); }

// shared-memory index of complex element c in the transpose planes: conflict-free for all four
// access patterns (phase A store / phase B load+store / phase C load), see DESIGN.md
LWB_HD int swz(int c)
{
    return c ^ (((c >> 5) & 1) | (((c >> 6) & 1) << 1) | (((c >> 4) & 1) << 2) |
                (((c >> 7) & 1) << 3) | (((c >> 8) & 1) << 4));
}

// Which complex element sits in (lane, slot, half) in each phase
LWB_HD int elemA(int lane, int slot, int half) { return (half ? 63 - lane : lane) + 64 * slot; }
LWB_HD int elemB(int lane, int slot, int half)
{
    return (((lane >> 3) * 2 + half) << 6) | (slot << 3) | (lane & 7);
}
LWB_HD int elemC(int lane, int slot, int half)
{
    const int T = half ? 63 - rev6(lane) : rev6(lane);
    return 8 * T + slot;
}
// output index m (0..511) of (lane, slot, half) AFTER the step-7 half swap of even slots
LWB_HD int outIndex(int lane, int slot, int half)
{
    const int flip = (slot & 1) ? half : !half;
    return 64 * rev3(slot) + (flip ? 63 - lane : lane);
}

// Host: build the per-lane pack from the blocksize-11 tables (a,b: 1024; c: 512; w: 1024).
inline void long_build_pack(const float *a, const float *b, const float *c, const float *w, float *pack)
{
    V *P = reinterpret_cast<V *>(pack);
    for (int lane = 0; lane < 32; lane++) {
        auto put = [&](int slot, float x, float y) { P[slot * 32 + lane] = V{x, y}; };
        float tx[2], ty[2];
        // phase A
        for (int j = 0; j < 8; j++) {
            for (int h = 0; h < 2; h++) {
                const int cc = elemA(lane, j, h);
                const float s = cc < 256 ? -1.0f : 1.0f;       // (-x)*A == x*(-A): sign moved into the table
                tx[h] = s * a[1022 - 2 * cc];
                ty[h] = s * a[1023 - 2 * cc];
            }
            put(P_S0W0 + j, tx[0], tx[1]);
            put(P_S0W1 + j, ty[0], ty[1]);
        }
        for (int j = 0; j < 4; j++) {
            for (int h = 0; h < 2; h++) {
                const int cc = elemA(lane, j, h);              // lower element of the step-2 butterfly
                tx[h] = a[1020 - 4 * cc];
                ty[h] = a[1021 - 4 * cc];
            }
            put(P_S2W0 + j, tx[0], tx[1]);
            put(P_S2W1 + j, ty[0], ty[1]);
        }
        for (int u = 0; u < 2; u++) {
            for (int h = 0; h < 2; h++) {
                const int r = (~elemA(lane, 2 + u, h)) & 127;  // stage 0: a = r * 8
                tx[h] = a[8 * r];
                ty[h] = a[8 * r + 1];
            }
            put(P_L0W0 + u, tx[0], tx[1]);
            put(P_L0W1 + u, ty[0], ty[1]);
        }
        for (int h = 0; h < 2; h++) {
            const int r = (~elemA(lane, 1, h)) & 63;           // stage 1: a = r * 16
            tx[h] = a[16 * r];
            ty[h] = a[16 * r + 1];
        }
        put(P_L1W0, tx[0], tx[1]);
        put(P_L1W1, ty[0], ty[1]);
        // phase B (both groups share the twiddle: same low bits)
        for (int u = 0; u < 4; u++) {
            const int r = (~elemB(lane, 4 + u, 0)) & 31;       // stage 2: a = r * 32
            put(P_L2W0 + u, a[32 * r], a[32 * r]);
            put(P_L2W1 + u, a[32 * r + 1], a[32 * r + 1]);
        }
        for (int u = 0; u < 2; u++) {
            const int r = (~elemB(lane, 2 + u, 0)) & 15;       // stage 3: a = r * 64
            put(P_L3W0 + u, a[64 * r], a[64 * r]);
            put(P_L3W1 + u, a[64 * r + 1], a[64 * r + 1]);
        }
        {
            const int r = (~elemB(lane, 1, 0)) & 7;            // stage 4: a = r * 128
            put(P_L4W0, a[128 * r], a[128 * r]);
            put(P_L4W1, a[128 * r + 1], a[128 * r + 1]);
        }
        // phase C
        put(P_A2, a[kLongN >> 3], a[kLongN >> 3]);
        for (int jj = 0; jj < 4; jj++) {
            for (int h = 0; h < 2; h++) {
                const int p = 511 - rev9(elemC(lane, 2 * jj + 1, h));   // step-7 index of the D side
                tx[h] = c[2 * p];
                ty[h] = c[2 * p + 1];
            }
            put(P_S7C0 + jj, tx[0], tx[1]);
            put(P_S7C1 + jj, ty[0], ty[1]);
        }
        for (int j = 0; j < 8; j++) {
            float b0[2], b1[2], wl[2], wh[2];
            for (int h = 0; h < 2; h++) {
                const int m = outIndex(lane, j, h);
                const int cp = 511 - m;                        // V element feeding output m
                b0[h] = b[2 * cp];
                b1[h] = b[2 * cp + 1];
                wl[h] = w[m];
                wh[h] = w[1023 - m];
            }
            put(P_B0 + j, b0[0], b0[1]);
            put(P_B1 + j, b1[0], b1[1]);
            put(P_WLO + j, wl[0], wl[1]);
            put(P_WHI + j, wh[0], wh[1]);
        }
    }
}

// ---- the per-lane arithmetic ----------------------------------------------------------------
// All phase functions are templated on NB = blocks a warp transforms in lockstep (1 or 2).  With
// NB = 2 every twiddle fetched from shared memory serves two independent blocks and the two
// instruction streams interleave, which is what hides the FP / shared-memory latencies at 12
// warps per SM (see DESIGN.md section 4.1).
struct Q4 { float x, y, z, w; };

LWB_HD Q4 ld_q4(const float *p)
{
#if defined(__CUDA_ARCH__)
    const float4 v = *reinterpret_cast<const float4 *>(p);
    return Q4{v.x, v.y, v.z, v.w};
#else
    return Q4{p[0], p[1], p[2], p[3]};
#endif
}

// step-3 butterfly (imdct.rs:36-41): hi/lo are complex values (O = odd index, E = even index)
LWB_HD void bfly(V &Oh, V &Eh, V &Ol, V &El, V w0, V w1)
{
    const V k00 = vsub(Oh, Ol);
    const V k01 = vsub(Eh, El);
    Oh = vadd(Oh, Ol);
    Eh = vadd(Eh, El);
    Ol = vsub_p(vmul(k00, w0), vmul(k01, w1));
    El = vadd_p(vmul(k01, w0), vmul(k00, w1));
}

// Phase A.  tile[b] = the block's 1024 spectrum floats.  Quad #f (4 floats at 4f) yields element
// c = f from (q1,q3) and c = 511-f from (q0,q2)  (step 0, imdct.rs:337-371).  The lane reads quads
// #(lane + 64 m) and #(63 - lane + 64 m), m < 4: they feed slots m and 7-m of both groups.
template <int NB, class TW>
LWB_HD void phase_a(const float *const tile[NB], int lane, TW tw, V O[NB][8], V E[NB][8])
{
#pragma unroll
    for (int m = 0; m < 4; m++) {
        Q4 f1[NB], f2[NB];
#pragma unroll
        for (int b = 0; b < NB; b++) {
            f1[b] = ld_q4(tile[b] + 4 * (lane + 64 * m));
            f2[b] = ld_q4(tile[b] + 4 * (63 - lane + 64 * m));
        }
        {
            const V w0 = tw(P_S0W0 + m), w1 = tw(P_S0W1 + m);
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const V qa = V{f1[b].w, f2[b].w}, qb = V{f1[b].y, f2[b].y};
                O[b][m] = vsub_p(vmul(qa, w0), vmul(qb, w1));
                E[b][m] = vadd_p(vmul(qa, w1), vmul(qb, w0));
            }
        }
        {
            const int j = 7 - m;
            const V w0 = tw(P_S0W0 + j), w1 = tw(P_S0W1 + j);
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const V qa = V{f2[b].x, f1[b].x}, qb = V{f2[b].z, f1[b].z};
                O[b][j] = vsub_p(vmul(qa, w0), vmul(qb, w1));
                E[b][j] = vadd_p(vmul(qa, w1), vmul(qb, w0));
            }
        }
    }
    // step 2 (imdct.rs:385-430): bit 8
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const V w0 = tw(P_S2W0 + j), w1 = tw(P_S2W1 + j);
#pragma unroll
        for (int b = 0; b < NB; b++) bfly(O[b][j + 4], E[b][j + 4], O[b][j], E[b][j], w0, w1);
    }
    // stage 0 (imdct.rs:445-446): bit 7
#pragma unroll
    for (int u = 0; u < 2; u++) {
        const V w0 = tw(P_L0W0 + u), w1 = tw(P_L0W1 + u);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            bfly(O[b][2 + u], E[b][2 + u], O[b][u], E[b][u], w0, w1);
            bfly(O[b][6 + u], E[b][6 + u], O[b][4 + u], E[b][4 + u], w0, w1);
        }
    }
    // stage 1 (imdct.rs:449-452): bit 6
    {
        const V w0 = tw(P_L1W0), w1 = tw(P_L1W1);
#pragma unroll
        for (int b = 0; b < NB; b++)
#pragma unroll
            for (int j = 1; j < 8; j += 2) bfly(O[b][j], E[b][j], O[b][j - 1], E[b][j - 1], w0, w1);
    }
}

// Phase B: stages 2,3,4 (imdct.rs:454-477): bits 5,4,3 = slot bits 2,1,0
template <int NB, class TW>
LWB_HD void phase_b(TW tw, V O[NB][8], V E[NB][8])
{
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const V w0 = tw(P_L2W0 + u), w1 = tw(P_L2W1 + u);
#pragma unroll
        for (int b = 0; b < NB; b++) bfly(O[b][4 + u], E[b][4 + u], O[b][u], E[b][u], w0, w1);
    }
#pragma unroll
    for (int u = 0; u < 2; u++) {
        const V w0 = tw(P_L3W0 + u), w1 = tw(P_L3W1 + u);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            bfly(O[b][2 + u], E[b][2 + u], O[b][u], E[b][u], w0, w1);
            bfly(O[b][6 + u], E[b][6 + u], O[b][4 + u], E[b][4 + u], w0, w1);
        }
    }
    {
        const V w0 = tw(P_L4W0), w1 = tw(P_L4W1);
#pragma unroll
        for (int b = 0; b < NB; b++)
#pragma unroll
            for (int j = 1; j < 8; j += 2) bfly(O[b][j], E[b][j], O[b][j - 1], E[b][j - 1], w0, w1);
    }
}

// imdct.rs:201-232 on slots s+3..s (z7[0] = O[s+3], z7[-1] = E[s+3], ...).  PROD: slots s+2 and
// s hold products (the ld654 multiplies by A[n/8]), so the four adds that read them use the
// never-contracted scalar form.
template <bool PROD>
LWB_HD void iter54(V O[8], V E[8], int s)
{
    const V k00 = vsub(O[s + 3], O[s + 1]);
    const V y0 = vadd(O[s + 3], O[s + 1]);
    const V y2 = PROD ? vadd_p(O[s + 2], O[s]) : vadd(O[s + 2], O[s]);
    const V k22 = PROD ? vsub_p(O[s + 2], O[s]) : vsub(O[s + 2], O[s]);
    O[s + 3] = vadd(y0, y2);
    O[s + 2] = vsub(y0, y2);
    const V k33 = PROD ? vsub_p(E[s + 2], E[s]) : vsub(E[s + 2], E[s]);
    O[s + 1] = vadd(k00, k33);
    O[s] = vsub(k00, k33);
    const V k11 = vsub(E[s + 3], E[s + 1]);
    const V y1 = vadd(E[s + 3], E[s + 1]);
    const V y3 = PROD ? vadd_p(E[s + 2], E[s]) : vadd(E[s + 2], E[s]);
    E[s + 3] = vadd(y1, y3);
    E[s + 2] = vsub(y1, y3);
    E[s + 1] = vsub(k11, k22);
    E[s] = vadd(k11, k22);
}

// ld654 (imdct.rs:234-288) for one block
LWB_HD void ld654(V O[8], V E[8], V a2)
{
    V k00, k11;
    k00 = vsub(O[7], O[3]); k11 = vsub(E[7], E[3]);
    O[7] = vadd(O[7], O[3]); E[7] = vadd(E[7], E[3]);
    O[3] = k00; E[3] = k11;
    k00 = vsub(O[6], O[2]); k11 = vsub(E[6], E[2]);
    O[6] = vadd(O[6], O[2]); E[6] = vadd(E[6], E[2]);
    O[2] = vmul(vadd(k00, k11), a2);
    E[2] = vmul(vsub(k11, k00), a2);
    k00 = vsub(O[1], O[5]); k11 = vsub(E[5], E[1]);
    O[5] = vadd(O[5], O[1]); E[5] = vadd(E[5], E[1]);
    O[1] = k11; E[1] = k00;
    k00 = vsub(O[0], O[4]); k11 = vsub(E[4], E[0]);
    O[4] = vadd(O[4], O[0]); E[4] = vadd(E[4], E[0]);
    O[0] = vmul(vadd(k00, k11), a2);
    E[0] = vmul(vsub(k00, k11), a2);
    iter54<false>(O, E, 4);
    iter54<true>(O, E, 0);
}

// Phase C part 1: ld654, then the half swap of the even slots and step 7 (imdct.rs:533-580).
// Steps 4-6 (imdct.rs:490-528) are pure renaming: U element 8T+j becomes V element
// 511 - rev9(8T+j) with (V.even, V.odd) = (U.odd, U.even) = (O, E).  Step 7 pairs V element p
// (odd slot j, "D") with 511-p (slot 7-j of the OTHER group, "E"): swapping the halves of the even
// slots lines partners up.  Afterwards slot j holds, per half, V element 511 - outIndex(..).
template <int NB, class TW>
LWB_HD void phase_c_fft(TW tw, V O[NB][8], V E[NB][8])
{
    const V a2 = tw(P_A2);
#pragma unroll
    for (int b = 0; b < NB; b++) {
        ld654(O[b], E[b], a2);
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            O[b][j] = V{O[b][j].y, O[b][j].x};
            E[b][j] = V{E[b][j].y, E[b][j].x};
        }
    }
#pragma unroll
    for (int jj = 0; jj < 4; jj++) {
        const int d = 2 * jj + 1, e = 7 - d;
        const V c0 = tw(P_S7C0 + jj), c1 = tw(P_S7C1 + jj);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const V a02 = vsub(O[b][d], O[b][e]);
            const V a11 = vadd(E[b][d], E[b][e]);
            const V b0 = vadd_p(vmul(c1, a02), vmul(c0, a11));
            const V b1 = vsub_p(vmul(c1, a11), vmul(c0, a02));
            const V b2 = vadd(O[b][d], O[b][e]);
            const V b3 = vsub(E[b][d], E[b][e]);
            O[b][d] = vadd(b2, b0);
            E[b][d] = vadd(b3, b1);
            O[b][e] = vsub(b2, b0);
            E[b][e] = vsub(b1, b3);
        }
    }
}

// Phase C part 2 for one slot of one block: step 8 (imdct.rs:589-658) + window/overlap-add
// (audio.rs:1112-1118).
//   p_odd  = out[m] = -out[1023-m];   p_even = out[1024+m] = out[2047-m]
//   pcm[m]      = p_odd * w[m] + prev[m] * w[1023-m]
//   pcm[1023-m] = (-p_odd) * w[1023-m] + prev[1023-m] * w[m]   (== prev*w[m] - p_odd*w[1023-m])
LWB_HD void step8_ola(V b0, V b1, V wlo, V whi, V Oj, V Ej, V prev_lo, V prev_hi, V &pcm_lo, V &pcm_hi, V &p_even)
{
    const V p_odd = vsub_p(vmul(Oj, b1), vmul(Ej, b0));
    p_even = vnsub_p(vmul(Oj, b0), vmul(Ej, b1));       // (-V.e)*B0 - V.o*B1, imdct.rs:620
    pcm_lo = vadd_p(vmul(p_odd, wlo), vmul(prev_lo, whi));
    pcm_hi = vsub_p(vmul(prev_hi, wlo), vmul(p_odd, whi));
}

#if defined(__CUDACC__)
// ---------------------------------------------------------------------------------------------
// device side
// ---------------------------------------------------------------------------------------------
#ifndef LWB_LONG_NB
#define LWB_LONG_NB 1
#endif
#ifndef LWB_LONG_WARPS
#define LWB_LONG_WARPS 8
#endif
#ifndef LWB_LONG_RING
#define LWB_LONG_RING (LWB_LONG_NB == 2 ? 2 : 5)
#endif
constexpr int kLongNB = LWB_LONG_NB;           // blocks (runs) a warp transforms in lockstep
constexpr int kLongWarps = LWB_LONG_WARPS;     // warps per CTA, one CTA per SM
constexpr int kLongRing = LWB_LONG_RING;       // ring stages per warp, each holding kLongNB tiles
constexpr int kLongTileBytes = kLongN2 * 4;
constexpr int kLongStageBytes = kLongNB * kLongTileBytes;
// [tiles: warps x ring x NB x 4 KB, 2 KB-aligned at run time][state tiles][pack][next-run descriptors][mbarriers]
constexpr size_t kLongSmemBytes = 2048 + (size_t)kLongWarps * (kLongRing + 1) * kLongStageBytes +
                                  (size_t)kLongPackFloats * 4 + kLongWarps * (kLongRing + 2) * 8 +
                                  kLongWarps * kLongNB * sizeof(LongRun) + 64;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    // try_wait suspends the warp until the phase completes or the hint (ns) expires, so a blocked
    // warp costs the scheduler almost no issue slots
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(200000u) : "memory");
}
// 1-D TMA: global -> shared, completion counted on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// transpose planes: E at [addr], O at [addr + 2048]
__device__ __forceinline__ void sts_eo(uint32_t addr, float e, float o)
{
    asm volatile("st.shared.f32 [%0], %1;\n\tst.shared.f32 [%0+2048], %2;" ::"r"(addr), "f"(e), "f"(o) : "memory");
}
__device__ __forceinline__ void lds_eo(uint32_t addr, float &e, float &o)
{
    asm volatile("ld.shared.f32 %0, [%2];\n\tld.shared.f32 %1, [%2+2048];" : "=f"(e), "=f"(o) : "r"(addr) : "memory");
}

// Twiddle residency: pack slots [kTwReg0, kTwReg1) live in registers for the whole kernel, the
// rest is read from the CTA's shared copy of the pack when used (compile-time choice per slot).
// Default (measured best on B200, profiles/variants_r1*.log): one block per warp, 8 warps per SM
// (2 per scheduler, 242 registers, no spills), a 5-tile ring, phase A / B / step-7 twiddles resident
// (slots 0..52) and the step-8 / window pairs fetched per block: 0.745 of the measured HBM peak.
// 12 warps x 164 registers with slots 16..29 resident: 0.734; 16 warps x 128 registers, nothing
// resident: 0.700; scalar instead of packed FP: -8 %; two blocks per warp (NB = 2) doubles the loop
// body past the instruction cache: 2x slower.
#ifndef LWB_TW_REG0
#define LWB_TW_REG0 0
#endif
#ifndef LWB_TW_REG1
#define LWB_TW_REG1 (LWB_LONG_NB == 2 ? 0 : 53)
#endif
constexpr int kTwReg0 = LWB_TW_REG0;
constexpr int kTwReg1 = LWB_TW_REG1;
struct TwMix {
    const V *r;                   // registers: slots [kTwReg0, kTwReg1)
    const V *lane_base;           // &pack[lane] in shared memory
    __device__ __forceinline__ V operator()(int slot) const
    {
        return (slot >= kTwReg0 && slot < kTwReg1) ? r[slot - kTwReg0] : lane_base[slot * 32];
    }
};

// Shared-memory byte offsets of the transposes: swz(elem(lane, slot, half)) * 4 splits into a
// lane part and a (slot, half) part combined by XOR (the tiles are 2 KB aligned, so the XOR can
// be applied to the full address): one LOP3 per access.
__device__ __forceinline__ uint32_t laneA(int lane, int half) { return 4u * (uint32_t)swz(elemA(lane, 0, half)); }
__device__ __forceinline__ uint32_t laneB(int lane) { return 4u * (uint32_t)swz(elemB(lane, 0, 0)); }
__device__ __forceinline__ uint32_t laneC(int lane, int half) { return 4u * (uint32_t)swz(elemC(lane, 0, half)); }
// compile-time (slot, half) parts: swz is XOR-linear, so swz(L ^ K) = swz(L) ^ swz(K) when L and K
// occupy disjoint bits of the element index
#define LWB_KA(j) (4u * (uint32_t)swz(64 * (j)))
#define LWB_KB(j, h) (4u * (uint32_t)swz(((h) << 6) | ((j) << 3)))
#define LWB_KC(j) (4u * (uint32_t)swz(j))

// Uniform (per-warp) view of the runs being processed
struct RunCur {
    const float *in;
    void *out;
    float *state;
    uint32_t in_stride;
    uint32_t flags;               // bit0 has_prev, bit1 write_state, bit2 dummy, bit3 first_short, bit4 last_short,
                                  // bit5 first_short == 2 (the left slope is exported, nothing is read from `state`)
};
__device__ __forceinline__ RunCur run_cur(const LongRun &r)
{
    return RunCur{r.in, r.out, r.state, r.in_stride,
                  (uint32_t)(r.has_prev ? 1u : 0u) | (r.write_state ? 2u : 0u) | (r.dummy ? 4u : 0u) |
                      (r.first_short ? 8u : 0u) | (r.last_short ? 16u : 0u)};
}
// k_long_s (one-pass schedule of mixed streams): a run may store its end state somewhere else than where it started from
struct RunCurS : RunCur { float *state_out; };
__device__ __forceinline__ RunCurS run_cur_s(const LongRun &r)
{
    RunCurS c;
    static_cast<RunCur &>(c) = run_cur(r);
    c.flags |= r.first_short == 2 ? 32u : 0u;
    c.state_out = r.state_out ? r.state_out : r.state;
    return c;
}

// samples.rs:92-103 (`Sample for i16`): x * 32768, clamp, truncate toward zero, NaN -> 0
__device__ __forceinline__ int16_t d_sample_i16(float v)
{
    // branch-free: cvt.rzi.s16.f32 truncates toward zero, clamps out-of-range inputs to the s16 range
    // (float-to-integer cvt saturates by definition) and turns NaN into 0; clamping after the
    // truncation equals clamping the float first (32767.x truncates to 32767, -32768.x to -32768).
    // (Pairing lanes to store two samples per 32-bit word was tried: the shuffles cost more than the
    // half-line stores, 471 vs 518 Gsamples/s, profiles/variants_r1k.log.)
    short r;
    asm("cvt.rzi.s16.f32 %0, %1;" : "=h"(r) : "f"(__fmul_rn(v, 32768.0f)));
    return (int16_t)r;
}
__device__ __forceinline__ void st_pcm(float *p, float v) { __stcs(p, v); }    // .cs beats .cg / default (variants_r1k.log)
__device__ __forceinline__ void st_pcm(int16_t *p, float v) { __stcs(reinterpret_cast<short *>(p), (short)d_sample_i16(v)); }

// Step 8 + window + overlap-add + stores, all 8 slots of all NB blocks.  FIRST: packet 0 of the
// run -- its previous right half comes from the stream state (staged in shared memory by TMA
// while the run's first tile was in flight) if has_prev, else nothing is emitted.  Streaming
// stores: PCM is written once and never read back by this kernel.
template <int NB, bool FIRST, typename OutT, typename RC = RunCur, int CS = 1>
__device__ __forceinline__ void out_stage(const TwMix &tw, int lane, const V O[NB][8], const V E[NB][8], V pe[NB][8],
                                          const RC cur[NB], OutT *out[NB], const float *s_state)
{
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int r64 = 64 * rev3(j);
        const bool nat = (j & 1);             // odd slots: half x -> lane, half y -> 63 - lane
        const V b0 = tw(P_B0 + j), b1 = tw(P_B1 + j);
        const V wlo = tw(P_WLO + j), whi = tw(P_WHI + j);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            V plo = pe[b][j], phi = pe[b][j];
            bool emit = !(cur[b].flags & 4u);
            if (FIRST) {
                emit = emit && (cur[b].flags & 1u);
                if (cur[b].flags & 1u) {
                    // prev[m] and prev[1023 - m] read separately: an imported state need not be symmetric
                    const float *s_lo = s_state + b * kLongN2 + lane, *s_hi = s_state + b * kLongN2 + 63 - lane;
                    const float ax = nat ? s_lo[r64] : s_hi[r64], ay = nat ? s_hi[r64] : s_lo[r64];
                    const float bx = nat ? s_hi[960 - r64] : s_lo[960 - r64];
                    const float by = nat ? s_lo[960 - r64] : s_hi[960 - r64];
                    plo = V{ax, ay};
                    phi = V{bx, by};
                }
            }
            V lo, hi, pev;
            step8_ola(b0, b1, wlo, whi, O[b][j], E[b][j], plo, phi, lo, hi, pev);
            pe[b][j] = pev;
            if (emit) {
                // m = r64 + lane (or + 63 - lane); 1023 - m = 960 - r64 + 63 - lane (or + lane)
                // (CS: samples between consecutive PCM elements of one channel -- 1 planar, C interleaved)
                OutT *o_lo = out[b] + lane * CS, *o_hi = out[b] + 63 * CS - lane * CS;
                if (nat) {
                    st_pcm(o_lo + r64 * CS, lo.x); st_pcm(o_hi + r64 * CS, lo.y);
                    st_pcm(o_hi + 960 * CS - r64 * CS, hi.x); st_pcm(o_lo + 960 * CS - r64 * CS, hi.y);
                } else {
                    st_pcm(o_hi + r64 * CS, lo.x); st_pcm(o_lo + r64 * CS, lo.y);
                    st_pcm(o_lo + 960 * CS - r64 * CS, hi.x); st_pcm(o_hi + 960 * CS - r64 * CS, hi.y);
                }
            }
        }
    }
}

__device__ __forceinline__ float lds_f32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}

// Packet 0 of a run that follows a short block (previous_window_flag == 0): the left window slope
// is the short one, centred in the left half (audio.rs:1059-1065 -> window_left_start = ls =
// (2048 - n0) / 4), the saved right half is pl = n0 / 2 samples long, and the packet emits
// x[ls .. 1024): pl windowed samples, then the rest of the left half as is (audio.rs:1112-1120).
// Rare (once per burst of short blocks), so plain scalar code; w = the short window slope.
// EXPORT: k_long_s -- runs may export their left slope (flags bit 5), and the slope is read from its shared-memory copy
// at w_s (through __ldg from global memory the four products of a lane each waited for an L2 round trip: 3.4 % of
// k_long_s's stall samples on the 6-channel config)
// LS: ls as a compile-time constant (0: use the argument) -- with it every position test below folds per slot.
template <int NB, typename OutT, typename RC = RunCur, bool EXPORT = false, int LS = 0, int CS = 1>
__device__ __forceinline__ void out_first_short(const TwMix &tw, int lane, const V O[NB][8], const V E[NB][8], V pe[NB][8],
                                                const RC cur[NB], OutT *out[NB], const float *s_state,
                                                const float *__restrict__ w, int ls_arg, uint32_t w_s = 0)
{
    const int ls = LS ? LS : ls_arg;
    const int pl = kLongN2 - 2 * ls;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int r64 = 64 * rev3(j);
        const bool nat = (j & 1);
        const V b0 = tw(P_B0 + j), b1 = tw(P_B1 + j);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const V p_odd = vsub_p(vmul(O[b][j], b1), vmul(E[b][j], b0));
            pe[b][j] = vnsub_p(vmul(O[b][j], b0), vmul(E[b][j], b1));
            if ((cur[b].flags & 5u) != 1u) continue;           // no history (or a dummy): nothing is emitted
            const float *prev = s_state + b * kLongN2;
            const bool exported = EXPORT && (cur[b].flags & 32u) != 0;     // the short block's kernel adds prev[i] w[pl-1-i] later
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const float po = h ? p_odd.y : p_odd.x;
                const int m = r64 + ((h == 0) == nat ? lane : 63 - lane);    // x[m] = p_odd, x[1023 - m] = -p_odd
                // x[m] lies on the slope iff m >= ls, and so does its mirror image (1023 - m - ls < pl <=> m >= ls); with
                // a compile-time ls that is a multiple of 64 the test is a property of the slot
                static_assert(LS % 64 == 0, "LS must be a multiple of 64");
                const bool on_slope = LS ? (r64 >= LS) : (m >= ls);
                if (on_slope) {
                    const int i = m - ls;                                      // < pl / 2
                    const float cw = __fmul_rn(po, (EXPORT ? lds_f32(w_s + 4u * (uint32_t)i) : __ldg(w + i)));
                    if (exported) cur[b].state[i] = cw;
                    else st_pcm(out[b] + i * CS, __fadd_rn(cw, __fmul_rn(prev[i], (EXPORT ? lds_f32(w_s + 4u * (uint32_t)(pl - 1 - i)) : __ldg(w + pl - 1 - i)))));
                }
                const int i = kLongN2 - 1 - m - ls;                            // >= pl / 2
                float v = -po;
                if (LS ? on_slope : (i < pl)) {
                    v = __fmul_rn(v, (EXPORT ? lds_f32(w_s + 4u * (uint32_t)i) : __ldg(w + i)));
                    if (exported) { cur[b].state[i] = v; continue; }
                    v = __fadd_rn(v, __fmul_rn(prev[i], (EXPORT ? lds_f32(w_s + 4u * (uint32_t)(pl - 1 - i)) : __ldg(w + pl - 1 - i))));
                }
                st_pcm(out[b] + i * CS, v);
            }
        }
    }
}

// runs: groups of kLongNB consecutive entries with equal n_packets (the host pads with dummy
// runs); pack: the twiddle pack of the setup's blocksize-11 tables (long_build_pack); ticket: a
// zeroed counter from which warps draw group indices.
//
// Latency plan per warp (lane 0 drives all asynchronous traffic; nothing below stalls the math):
//   * spectrum tiles: 1-D TMA into a ring, issued in processing order ACROSS run boundaries;
//   * the ticket for the next group is drawn (atomicAdd) when a group starts and first looked at
//     a packet later; its descriptors then arrive by TMA into shared memory;
//   * the stream state a run overlaps with (has_prev) arrives by TMA into a per-warp state tile
//     while the run's first spectrum tile is in flight.
// CS: PCM step of a channel (1: planar; C: interleaved, one instantiation per channel count so that every store
// offset stays an immediate and the planar instantiations keep their code)
template <typename OutT, int CS = 1>
__global__ void __launch_bounds__(kLongWarps * 32, 1)
k_long(const LongRun *__restrict__ runs, uint32_t n_groups, const float *__restrict__ pack,
       unsigned int *__restrict__ ticket, const float *__restrict__ w_short, int ls)
{
    constexpr int NB = kLongNB;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // tiles first, aligned to 2 KB in the shared window
    const uint32_t raw_s = smem_u32(smem_raw);
    const uint32_t align_pad = (2048u - (raw_s & 2047u)) & 2047u;
    unsigned char *base = smem_raw + align_pad;
    constexpr size_t kTilesBytes = (size_t)kLongWarps * kLongRing * kLongStageBytes;
    constexpr size_t kStateBytes = (size_t)kLongWarps * kLongStageBytes;
    float *tiles = reinterpret_cast<float *>(base) + (size_t)warp * kLongRing * NB * kLongN2;
    float *s_state = reinterpret_cast<float *>(base + kTilesBytes) + (size_t)warp * NB * kLongN2;
    V *s_pack = reinterpret_cast<V *>(base + kTilesBytes + kStateBytes);
    unsigned char *tail = base + kTilesBytes + kStateBytes + (size_t)kLongPackFloats * 4;
    LongRun *s_next = reinterpret_cast<LongRun *>(tail) + warp * NB;                       // 16-aligned
    uint64_t *bars = reinterpret_cast<uint64_t *>(tail + (size_t)kLongWarps * NB * sizeof(LongRun)) +
                     warp * (kLongRing + 2);
    if (n_groups == 0) return;

    // stage the pack once per CTA
    {
        const float4 *src = reinterpret_cast<const float4 *>(pack);
        float4 *dst = reinterpret_cast<float4 *>(s_pack);
        for (int i = threadIdx.x; i < kLongPackFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    if (lane == 0) {
        for (int i = 0; i < kLongRing + 2; i++) mbar_init(smem_u32(&bars[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    V twR[kTwReg1 - kTwReg0 > 0 ? kTwReg1 - kTwReg0 : 1];
#pragma unroll
    for (int s = kTwReg0; s < kTwReg1; s++) twR[s - kTwReg0] = s_pack[s * 32 + lane];
    const TwMix tw{twR, s_pack + lane};

    const uint32_t tiles_s = smem_u32(tiles);
    const uint32_t bars_s = smem_u32(bars);
    const uint32_t bar_state = bars_s + 8 * kLongRing, bar_desc = bars_s + 8 * (kLongRing + 1);
    const uint32_t state_s = smem_u32(s_state), next_s = smem_u32(s_next);
    const uint32_t lA0 = laneA(lane, 0), lA1 = laneA(lane, 1);
    const uint32_t lB = laneB(lane);
    const uint32_t lC0 = laneC(lane, 0), lC1 = laneC(lane, 1);
    uint32_t phase_bits = 0;                  // bit i: parity of ring stage i; bits 30/31: state / descriptor barrier
    uint32_t slot_i = 0;                      // ring stage of the packets being processed

    // lane 0's cursor over the asynchronous traffic
    uint32_t lc = 0;                          // stages of the current group issued so far
    uint32_t nx_idx = 0;                      // ticket drawn for the next group (value used a packet later)
    uint32_t nx_stage = 0;                    // 0 ticket drawn, 1 descriptor in flight, 2 descriptor landed, 3 none
    uint32_t nx_lc = 0, nx_npk = 0;
    uint32_t nx_state_issued = 0;             // next group's state tile already requested
    uint32_t desc_parity = 0;
    RunCur cur[NB];
    uint32_t npk;

    auto issue_stage = [&](uint32_t stage, const LongRun *r, uint32_t pkt) {     // lane 0 only
        const uint32_t bar = bars_s + 8 * stage;
        mbar_expect_tx(bar, kLongStageBytes);
#pragma unroll
        for (int b = 0; b < NB; b++)
            tma_load_1d(tiles_s + stage * kLongStageBytes + b * kLongTileBytes,
                        r[b].in + (size_t)pkt * r[b].in_stride, kLongTileBytes, bar);
    };
    auto issue_stage_cur = [&](uint32_t stage, uint32_t pkt) {                   // lane 0 only
        const uint32_t bar = bars_s + 8 * stage;
        mbar_expect_tx(bar, kLongStageBytes);
#pragma unroll
        for (int b = 0; b < NB; b++)
            tma_load_1d(tiles_s + stage * kLongStageBytes + b * kLongTileBytes,
                        cur[b].in + (size_t)pkt * cur[b].in_stride, kLongTileBytes, bar);
    };
    // request the state rows of a group (lane 0 only).  Every group arms the barrier exactly once
    // (with 0 bytes if none of its runs has history) so that the parity bookkeeping stays uniform.
    auto issue_state = [&](const float *const st[NB], const uint32_t has[NB]) {
        uint32_t bytes = 0;
#pragma unroll
        for (int b = 0; b < NB; b++) bytes += has[b] ? kLongTileBytes : 0;
        mbar_expect_tx(bar_state, bytes);
#pragma unroll
        for (int b = 0; b < NB; b++)
            if (has[b]) tma_load_1d(state_s + b * kLongTileBytes, st[b], kLongTileBytes, bar_state);
    };

    {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(ticket, 1u);
        idx = __shfl_sync(0xffffffffu, idx, 0);
        if (idx >= n_groups) return;
#pragma unroll
        for (int b = 0; b < NB; b++) cur[b] = run_cur(runs[idx * NB + b]);
        npk = runs[idx * NB].n_packets;
        if (lane == 0) {
            fence_proxy_async();
            const float *st[NB];
            uint32_t has[NB];
#pragma unroll
            for (int b = 0; b < NB; b++) { st[b] = cur[b].state; has[b] = cur[b].flags & 1u; }
            issue_state(st, has);
            for (; lc < (uint32_t)kLongRing && lc < npk; lc++) issue_stage_cur(lc, lc);
            nx_idx = atomicAdd(ticket, 1u);            // not looked at before the next packet
        }
    }

    for (;;) {
        V pe[NB][8];
#pragma unroll
        for (int b = 0; b < NB; b++)
#pragma unroll
            for (int j = 0; j < 8; j++) pe[b][j] = V{0.f, 0.f};
        OutT *out[NB];
#pragma unroll
        for (int b = 0; b < NB; b++) out[b] = static_cast<OutT *>(cur[b].out);

        for (uint32_t p = 0; p < npk; p++) {
            const uint32_t stage_s = tiles_s + slot_i * kLongStageBytes;
            mbar_wait(bars_s + 8 * slot_i, (phase_bits >> slot_i) & 1u);
            phase_bits ^= 1u << slot_i;

            V O[NB][8], E[NB][8];
            {
                const float *tp[NB];
#pragma unroll
                for (int b = 0; b < NB; b++) tp[b] = tiles + (slot_i * NB + b) * kLongN2;
                phase_a<NB>(tp, lane, tw, O, E);
            }
            __syncwarp();           // every lane has consumed its quads: the tiles become the scratch
            // transpose 1 (per block: E plane | O plane in its own tile)
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const uint32_t t = stage_s + b * kLongTileBytes;
                const uint32_t a0 = t + lA0, a1 = t + lA1;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    sts_eo(a0 ^ LWB_KA(j), E[b][j].x, O[b][j].x);
                    sts_eo(a1 ^ LWB_KA(j), E[b][j].y, O[b][j].y);
                }
            }
            __syncwarp();
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const uint32_t b0 = stage_s + b * kLongTileBytes + lB;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    lds_eo(b0 ^ LWB_KB(j, 0), E[b][j].x, O[b][j].x);
                    lds_eo(b0 ^ LWB_KB(j, 1), E[b][j].y, O[b][j].y);
                }
            }
            __syncwarp();
            phase_b<NB>(tw, O, E);
            // transpose 2
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const uint32_t b0 = stage_s + b * kLongTileBytes + lB;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    sts_eo(b0 ^ LWB_KB(j, 0), E[b][j].x, O[b][j].x);
                    sts_eo(b0 ^ LWB_KB(j, 1), E[b][j].y, O[b][j].y);
                }
            }
            __syncwarp();
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const uint32_t t = stage_s + b * kLongTileBytes;
                const uint32_t c0 = t + lC0, c1 = t + lC1;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    lds_eo(c0 ^ LWB_KC(j), E[b][j].x, O[b][j].x);
                    lds_eo(c1 ^ LWB_KC(j), E[b][j].y, O[b][j].y);
                }
            }
            __syncwarp();
            // the stage is free again: refill it with the next tiles in processing order
            if (lane == 0) {
                if (nx_stage == 0 && p >= 1) {          // the ticket drawn a packet ago has long arrived
                    if (nx_idx < n_groups) {
                        fence_proxy_async();
                        mbar_expect_tx(bar_desc, NB * (uint32_t)sizeof(LongRun));
                        tma_load_1d(next_s, runs + (size_t)nx_idx * NB, NB * (uint32_t)sizeof(LongRun), bar_desc);
                        nx_stage = 1;
                    } else {
                        nx_stage = 3;
                    }
                }
                // Stages are filled strictly in processing order: `ahead` tiles are in flight behind the
                // one just consumed, in stages slot_i+1 .. slot_i+ahead, so the next tile goes to
                // slot_i+1+ahead (== slot_i once the ring is full).  One tile per packet: a ring left
                // under-filled by groups shorter than itself is topped up at the next hand-over (a
                // catch-up loop here costs 2-9% of the steady state, profiles/variants_r1k.log).
                uint32_t ahead = lc - (p + 1) + nx_lc;
                if (ahead < (uint32_t)kLongRing) {
                    uint32_t tgt = slot_i + 1 + ahead;
                    if (tgt >= (uint32_t)kLongRing) tgt -= kLongRing;
                    if (lc < npk) {
                        fence_proxy_async();
                        issue_stage_cur(tgt, lc);
                        lc++;
                    } else {
                        if (nx_stage == 1) {
                            mbar_wait(bar_desc, desc_parity);
                            desc_parity ^= 1u;
                            nx_stage = 2;
                            nx_npk = s_next[0].n_packets;
                            nx_lc = 0;
                        }
                        if (nx_stage == 2 && nx_lc < nx_npk) {
                            fence_proxy_async();
                            issue_stage(tgt, s_next, nx_lc);
                            nx_lc++;
                        }
                    }
                }
            }
            phase_c_fft<NB>(tw, O, E);
            if (p > 0) {
                out_stage<NB, false, OutT, RunCur, CS>(tw, lane, O, E, pe, cur, out, s_state);
            } else {
                mbar_wait(bar_state, (phase_bits >> 30) & 1u);      // armed once per group
                phase_bits ^= 1u << 30;
                if (NB == 1 && (cur[0].flags & 8u))
                    out_first_short<NB, OutT, RunCur, false, 0, CS>(tw, lane, O, E, pe, cur, out, s_state, w_short, ls);
                else
                    out_stage<NB, true, OutT, RunCur, CS>(tw, lane, O, E, pe, cur, out, s_state);
                __syncwarp();                                       // state tile consumed
            }
#pragma unroll
            for (int b = 0; b < NB; b++)
                if (p > 0 || (cur[b].flags & 1u)) out[b] += ((p == 0 && (cur[b].flags & 8u)) ? kLongN2 - ls : kLongN2) * CS;
            // the state tile is free after packet 0: request the next group's state rows as soon as
            // its descriptors are known
            if (lane == 0 && nx_stage == 2 && !nx_state_issued) {
                const float *st[NB];
                uint32_t has[NB];
#pragma unroll
                for (int b = 0; b < NB; b++) { st[b] = s_next[b].state; has[b] = s_next[b].has_prev; }
                fence_proxy_async();
                issue_state(st, has);
                nx_state_issued = 1;
            }
            slot_i = (slot_i + 1 == (uint32_t)kLongRing) ? 0 : slot_i + 1;
        }
#pragma unroll
        for (int b = 0; b < NB; b++) {
            if ((cur[b].flags & 16u)) {
                // the last packet precedes a short block (next_window_flag == 0, audio.rs:1067-1073):
                // window_right_start = 1024 + ls, so x[1024 .. 1024 + ls) leaves with this packet and the
                // pl samples after them are what the short block overlaps with
                const bool emitted = (npk > 1 || (cur[b].flags & 1u)) && !(cur[b].flags & 4u);
                const bool keep = (cur[b].flags & 6u) == 2u;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int r64 = 64 * rev3(j);
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const float v = ((j & 1) != 0) == (h == 0) ? pe[b][j].x : pe[b][j].y;
                        const int m = r64 + (h ? 63 - lane : lane);          // x[1024 + m] = x[2047 - m] = v
                        if (m < ls) {
                            if (emitted) st_pcm(out[b] + m * CS, v);
                        } else if (keep && m < kLongN2 - ls) {      // the pl = 1024 - 2 ls samples the short block overlaps with
                            cur[b].state[m - ls] = v;
                            cur[b].state[kLongN2 - 1 - ls - m] = v;
                        }
                    }
                }
            } else if ((cur[b].flags & 6u) == 2u) {       // write_state and not dummy
                float *s_lo = cur[b].state + lane, *s_hi = cur[b].state + 63 - lane;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int r64 = 64 * rev3(j);
                    const float vx = (j & 1) ? pe[b][j].x : pe[b][j].y, vy = (j & 1) ? pe[b][j].y : pe[b][j].x;
                    s_lo[r64] = vx; s_hi[r64] = vy;                 // state[m]
                    s_hi[960 - r64] = vx; s_lo[960 - r64] = vy;     // state[1023 - m]: same value (imdct.rs:622-649)
                }
            }
        }
        // hand over to the group lane 0 has (maybe) already started loading.  Short groups can get
        // here before the asynchronous steps ran: finish them synchronously.
        uint32_t st_ = 0, nlc = 0;
        if (lane == 0) {
            if (nx_stage == 0) {
                if (nx_idx < n_groups) {
                    fence_proxy_async();
                    mbar_expect_tx(bar_desc, NB * (uint32_t)sizeof(LongRun));
                    tma_load_1d(next_s, runs + (size_t)nx_idx * NB, NB * (uint32_t)sizeof(LongRun), bar_desc);
                    nx_stage = 1;
                } else {
                    nx_stage = 3;
                }
            }
            if (nx_stage == 1) {
                mbar_wait(bar_desc, desc_parity);
                desc_parity ^= 1u;
                nx_stage = 2;
                nx_npk = s_next[0].n_packets;
                nx_lc = 0;
            }
            if (nx_stage == 2 && !nx_state_issued) {
                const float *st[NB];
                uint32_t has[NB];
#pragma unroll
                for (int b = 0; b < NB; b++) { st[b] = s_next[b].state; has[b] = s_next[b].has_prev; }
                fence_proxy_async();
                issue_state(st, has);
            }
            st_ = nx_stage;
            nlc = nx_lc;
        }
        st_ = __shfl_sync(0xffffffffu, st_, 0);
        nlc = __shfl_sync(0xffffffffu, nlc, 0);
        if (st_ != 2) break;
        // lane 0 has acquired the descriptor tile through its mbarrier wait; the warp barrier extends that
        // to the other lanes (a shuffle alone is not a memory-ordering operation).  Letting every lane
        // wait on the mbarrier itself costs 2 % (code layout), profiles/variants_r1k.log.
        __syncwarp();
#pragma unroll
        for (int b = 0; b < NB; b++) cur[b] = run_cur(s_next[b]);
        npk = s_next[0].n_packets;
        __syncwarp();                              // s_next may be overwritten from here on
        lc = nlc;
        nx_stage = 0; nx_lc = 0; nx_npk = 0; nx_state_issued = 0;
        if (lane == 0) {
            // top the ring up (new group longer than what was prefetched so far)
            fence_proxy_async();
            for (uint32_t k = lc; k < (uint32_t)kLongRing && k < npk; k++) {
                issue_stage_cur((slot_i + k) % kLongRing, k);
                lc = k + 1;
            }
            nx_idx = atomicAdd(ticket, 1u);        // ticket for the group after this one
        }
    }
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------------------------------------------------------------------------------------
// k_long_s: the same transform behind a different driver, for launches made of MANY SHORT runs (the one-pass
// schedule of mixed long / short streams, path_mixed.cuh: a run is what lies between two bursts of short
// blocks, often one to three packets).  k_long learns its next group one group ahead (ticket, then descriptor,
// then tiles), which leaves the ring under-filled and the descriptor latency exposed when groups are shorter
// than the ring.  Here the deal is static (run r -> warp r mod W), so a warp knows its whole future:
//   * descriptors arrive by cp.async in a shared ring, kLongFetch runs ahead of the producer;
//   * the producer cursor walks (run, packet) in processing order and stays exactly kLongRing tiles ahead of
//     the consumer, across any number of run boundaries;
//   * the state row of the next run that overlaps with one (has_prev, not exported) is requested as soon as the
//     state tile is free and that run's descriptor has landed.
// ---------------------------------------------------------------------------------------------
constexpr int kLongLs256 = (kLongN - 256) / 4;      // ls of a long block next to a 256-point block
constexpr int kLongFetch = 3;
constexpr int kLongDescSlots = kLongFetch + kLongRing + 3;
constexpr int kLongSlopeMax = 512;       // floats of the short window slope kept in shared memory (blocksize_0 <= 1024)
constexpr size_t kLongSmemBytesS = 2048 + (size_t)kLongWarps * (kLongRing + 1) * kLongTileBytes + (size_t)kLongPackFloats * 4 +
                                   kLongWarps * (kLongRing + 2) * 8 + (size_t)kLongWarps * kLongDescSlots * sizeof(LongRun) +
                                   kLongSlopeMax * sizeof(float) + 64;

template <typename OutT, int LS>
__global__ void __launch_bounds__(kLongWarps * 32, 1)
k_long_s(const LongRun *__restrict__ runs, uint32_t n_runs, const float *__restrict__ pack,
         const float *__restrict__ w_short, int ls_arg)
{
    constexpr int NB = 1;
    const int ls = LS ? LS : ls_arg;          // LS = 448: blocksize_0 = 256, the only short size the one-pass schedule has
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t raw_s = smem_u32(smem_raw);
    const uint32_t align_pad = (2048u - (raw_s & 2047u)) & 2047u;
    unsigned char *base = smem_raw + align_pad;
    constexpr size_t kTilesBytes = (size_t)kLongWarps * kLongRing * kLongTileBytes;
    constexpr size_t kStateBytes = (size_t)kLongWarps * kLongTileBytes;
    float *tiles = reinterpret_cast<float *>(base) + (size_t)warp * kLongRing * kLongN2;
    float *s_state = reinterpret_cast<float *>(base + kTilesBytes) + (size_t)warp * kLongN2;
    V *s_pack = reinterpret_cast<V *>(base + kTilesBytes + kStateBytes);
    unsigned char *tail = base + kTilesBytes + kStateBytes + (size_t)kLongPackFloats * 4;
    LongRun *s_desc = reinterpret_cast<LongRun *>(tail) + warp * kLongDescSlots;               // 16-aligned
    uint64_t *bars = reinterpret_cast<uint64_t *>(tail + (size_t)kLongWarps * kLongDescSlots * sizeof(LongRun)) + warp * (kLongRing + 2);
    float *s_w = reinterpret_cast<float *>(tail + (size_t)kLongWarps * kLongDescSlots * sizeof(LongRun) + (size_t)kLongWarps * (kLongRing + 2) * 8);
    {
        const int pl = kLongN2 - 2 * ls;                     // the short slope: pl floats (0 when no run of the launch needs it)
        if (w_short)                                         // (pl <= kLongSlopeMax: the host checks)
            for (int i = threadIdx.x; i < pl && i < kLongSlopeMax; i += blockDim.x) s_w[i] = __ldg(w_short + i);
    }
    const uint32_t w_s = smem_u32(s_w);
    {
        const float4 *src = reinterpret_cast<const float4 *>(pack);
        float4 *dst = reinterpret_cast<float4 *>(s_pack);
        for (int i = threadIdx.x; i < kLongPackFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    if (lane == 0) {
        for (int i = 0; i < kLongRing + 1; i++) mbar_init(smem_u32(&bars[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    V twR[kTwReg1 - kTwReg0 > 0 ? kTwReg1 - kTwReg0 : 1];
#pragma unroll
    for (int s = kTwReg0; s < kTwReg1; s++) twR[s - kTwReg0] = s_pack[s * 32 + lane];
    const TwMix tw{twR, s_pack + lane};

    const uint32_t tiles_s = smem_u32(tiles), bars_s = smem_u32(bars), desc_s = smem_u32(s_desc);
    const uint32_t bar_state = bars_s + 8 * kLongRing, state_s = smem_u32(s_state);
    const uint32_t lA0 = laneA(lane, 0), lA1 = laneA(lane, 1);
    const uint32_t lB = laneB(lane);
    const uint32_t lC0 = laneC(lane, 0), lC1 = laneC(lane, 1);

    const uint32_t W = gridDim.x * kLongWarps, gw = blockIdx.x * kLongWarps + warp;
    if (gw >= n_runs) return;
    const uint4 *rq = reinterpret_cast<const uint4 *>(runs);
    uint32_t f_run = gw, f_slot = 0;
    auto fetch = [&]() {            // cp.async groups are per thread: lanes 0..2 copy one quad each, everybody commits / waits
        if (lane < 3 && f_run < n_runs) cp_async16(desc_s + f_slot * (uint32_t)sizeof(LongRun) + lane * 16, rq + 3 * (size_t)f_run + lane);
        cp_async_commit();
        f_run += W;
        f_slot = (f_slot + 1 == (uint32_t)kLongDescSlots) ? 0 : f_slot + 1;
    };
#pragma unroll
    for (int i = 0; i <= kLongFetch; i++) fetch();
    cp_async_wait<kLongFetch>();
    __syncwarp();
    // ---- producer (warp-uniform cursor; lane 0 issues) ----
    uint32_t p_run = gw, p_pkt = 0, p_slot = 0, p_stage = 0;
    const float *p_in = s_desc[0].in;
    uint32_t p_stride = s_desc[0].in_stride, p_npk = s_desc[0].n_packets;
    auto produce = [&]() {
        if (lane == 0) {
            fence_proxy_async();          // the stage was written through the generic proxy (transposes) before
            const uint32_t bar = bars_s + 8 * p_stage;
            mbar_expect_tx(bar, kLongTileBytes);
            tma_load_1d(tiles_s + p_stage * kLongTileBytes, p_in + (size_t)p_pkt * p_stride, kLongTileBytes, bar);
        }
        p_stage = (p_stage + 1 == (uint32_t)kLongRing) ? 0 : p_stage + 1;
        if (++p_pkt >= p_npk) {
            p_run += W;
            p_pkt = 0;
            p_slot = (p_slot + 1 == (uint32_t)kLongDescSlots) ? 0 : p_slot + 1;
            fetch();                      // run p_run + kLongFetch * W
            cp_async_wait<kLongFetch>();  // run p_run's descriptor has landed
            __syncwarp();
            if (p_run < n_runs) { p_in = s_desc[p_slot].in; p_stride = s_desc[p_slot].in_stride; p_npk = s_desc[p_slot].n_packets; }
        }
    };
    for (int i = 0; i < kLongRing; i++)
        if (p_run < n_runs) produce();

    // ---- state rows: st_run = the run whose row is in the tile or on its way (~0: the tile is free) ----
    uint32_t st_run = ~0u;
    auto issue_state = [&](const float *row, uint32_t run) {
        if (lane == 0) {
            fence_proxy_async();
            mbar_expect_tx(bar_state, kLongTileBytes);
            tma_load_1d(state_s, row, kLongTileBytes, bar_state);
        }
        st_run = run;
    };
    // first run in [from_run, p_run] that reads a row; the descriptor slots between the consumer and the producer have
    // landed and are not overwritten before the consumer has passed them
    auto request_state = [&](uint32_t from_run, uint32_t from_slot) {
        uint32_t r = from_run, sl = from_slot;
        while (r < n_runs && r <= p_run) {
            const LongRun &d = s_desc[sl];
            if (d.has_prev && d.first_short != 2) {
                issue_state(d.state, r);
                return;
            }
            r += W;
            sl = (sl + 1 == (uint32_t)kLongDescSlots) ? 0 : sl + 1;
        }
    };

    uint32_t phase_bits = 0, slot_i = 0, c_slot = 0;
    for (uint32_t c_run = gw; c_run < n_runs; c_run += W) {
        RunCurS cur[NB];
        cur[0] = run_cur_s(s_desc[c_slot]);
        const uint32_t npk = s_desc[c_slot].n_packets;
        const uint32_t my_slot = c_slot;
        c_slot = (c_slot + 1 == (uint32_t)kLongDescSlots) ? 0 : c_slot + 1;
        const bool need_state = (cur[0].flags & 33u) == 1u;
        if (st_run == ~0u) request_state(c_run, my_slot);
        V pe[NB][8];
#pragma unroll
        for (int j = 0; j < 8; j++) pe[0][j] = V{0.f, 0.f};
        OutT *out[NB];
        out[0] = static_cast<OutT *>(cur[0].out);

        for (uint32_t p = 0; p < npk; p++) {
            const uint32_t stage_s = tiles_s + slot_i * kLongTileBytes;
            mbar_wait(bars_s + 8 * slot_i, (phase_bits >> slot_i) & 1u);
            phase_bits ^= 1u << slot_i;
            V O[NB][8], E[NB][8];
            {
                const float *tp[NB];
                tp[0] = tiles + slot_i * kLongN2;
                phase_a<NB>(tp, lane, tw, O, E);
            }
            __syncwarp();           // every lane has consumed its quads: the tile becomes the scratch
            {
                const uint32_t a0 = stage_s + lA0, a1 = stage_s + lA1;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    sts_eo(a0 ^ LWB_KA(j), E[0][j].x, O[0][j].x);
                    sts_eo(a1 ^ LWB_KA(j), E[0][j].y, O[0][j].y);
                }
            }
            __syncwarp();
            {
                const uint32_t b0 = stage_s + lB;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    lds_eo(b0 ^ LWB_KB(j, 0), E[0][j].x, O[0][j].x);
                    lds_eo(b0 ^ LWB_KB(j, 1), E[0][j].y, O[0][j].y);
                }
            }
            __syncwarp();
            phase_b<NB>(tw, O, E);
            {
                const uint32_t b0 = stage_s + lB;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    sts_eo(b0 ^ LWB_KB(j, 0), E[0][j].x, O[0][j].x);
                    sts_eo(b0 ^ LWB_KB(j, 1), E[0][j].y, O[0][j].y);
                }
            }
            __syncwarp();
            {
                const uint32_t c0 = stage_s + lC0, c1 = stage_s + lC1;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    lds_eo(c0 ^ LWB_KC(j), E[0][j].x, O[0][j].x);
                    lds_eo(c1 ^ LWB_KC(j), E[0][j].y, O[0][j].y);
                }
            }
            __syncwarp();
            if (p_run < n_runs) produce();          // the stage is free again
            phase_c_fft<NB>(tw, O, E);
            if (p > 0) {
                out_stage<NB, false, OutT, RunCurS>(tw, lane, O, E, pe, cur, out, s_state);
            } else {
                if (need_state) {
                    if (st_run != c_run) issue_state(cur[0].state, c_run);  // (its descriptor had not landed when the tile came free)
                    mbar_wait(bar_state, (phase_bits >> 30) & 1u);
                    phase_bits ^= 1u << 30;
                }
                if (cur[0].flags & 8u)
                    out_first_short<NB, OutT, RunCurS, true, LS>(tw, lane, O, E, pe, cur, out, s_state, w_short, ls, w_s);
                else
                    out_stage<NB, true, OutT, RunCurS>(tw, lane, O, E, pe, cur, out, s_state);
                __syncwarp();
                if (need_state) {                                           // state tile consumed: on to the next run that needs it
                    st_run = ~0u;
                    request_state(c_run + W, c_slot);
                }
            }
            if (p > 0 || (cur[0].flags & 1u)) out[0] += (p == 0 && (cur[0].flags & 8u)) ? kLongN2 - ls : kLongN2;
            slot_i = (slot_i + 1 == (uint32_t)kLongRing) ? 0 : slot_i + 1;
        }
        if ((cur[0].flags & 16u)) {
            // the last packet precedes a short block: see k_long
            const bool emitted = (npk > 1 || (cur[0].flags & 1u)) && !(cur[0].flags & 4u);
            const bool keep = (cur[0].flags & 6u) == 2u;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int r64 = 64 * rev3(j);
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const float v = ((j & 1) != 0) == (h == 0) ? pe[0][j].x : pe[0][j].y;
                    const int m = r64 + (h ? 63 - lane : lane);          // x[1024 + m] = x[2047 - m] = v
                    const bool before = LS ? (r64 < LS) : (m < ls);      // (a multiple of 64: a property of the slot)
                    if (before) {
                        if (emitted) st_pcm(out[0] + m, v);
                    } else if (keep && m < kLongN2 - ls) {
                        cur[0].state_out[m - ls] = v;
                        cur[0].state_out[kLongN2 - 1 - ls - m] = v;
                    }
                }
            }
        } else if ((cur[0].flags & 6u) == 2u) {
            float *s_lo = cur[0].state_out + lane, *s_hi = cur[0].state_out + 63 - lane;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int r64 = 64 * rev3(j);
                const float vx = (j & 1) ? pe[0][j].x : pe[0][j].y, vy = (j & 1) ? pe[0][j].y : pe[0][j].x;
                s_lo[r64] = vx; s_hi[r64] = vy;
                s_hi[960 - r64] = vx; s_lo[960 - r64] = vy;
            }
        }
    }
}

inline int long_launch_static(cudaStream_t stream, const LongRun *d_runs, uint32_t n_runs, const float *d_pack, int sm_count,
                              bool i16_out, const float *d_w_short, int ls)
{
    if (!n_runs) return 0;
    const uint32_t want = (n_runs + kLongWarps - 1) / kLongWarps;
    const uint32_t grid = want < (uint32_t)sm_count ? want : (uint32_t)sm_count;
    // only blocksize_0 = 256 is instantiated: it is the one short size the one-pass schedule exists for (k_short), and
    // the runtime-ls variant of this kernel makes ptxas 12.9 crash
    if (ls != kLongLs256) return 1;
    if (i16_out) k_long_s<int16_t, kLongLs256><<<grid, kLongWarps * 32, kLongSmemBytesS, stream>>>(d_runs, n_runs, d_pack, d_w_short, ls);
    else k_long_s<float, kLongLs256><<<grid, kLongWarps * 32, kLongSmemBytesS, stream>>>(d_runs, n_runs, d_pack, d_w_short, ls);
    return cudaGetLastError() != cudaSuccess;
}

// The k_long instantiations: planar (CS = 1) and interleaved for 2..8 channels, f32 and i16.
#define LWB_LONG_STEPS(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)

inline void long_kernel_configure()
{
#define LWB_LONG_CONF(CS)                                                                                      \
    cudaFuncSetAttribute(k_long<float, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLongSmemBytes); \
    cudaFuncSetAttribute(k_long<int16_t, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLongSmemBytes);
    LWB_LONG_STEPS(LWB_LONG_CONF)
#undef LWB_LONG_CONF
    cudaFuncSetAttribute(k_long_s<float, kLongLs256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLongSmemBytesS);
    cudaFuncSetAttribute(k_long_s<int16_t, kLongLs256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLongSmemBytesS);
}

// d_runs: n_groups * kLongNB descriptors.  Returns 0 on success; `ticket` must point at a zeroed
// device word no other launch in flight uses.  step: PCM elements between consecutive samples of
// one channel -- 1 for planar output, the channel count (2..8) for interleaved output.
inline int long_launch(cudaStream_t stream, const LongRun *d_runs, uint32_t n_groups, const float *d_pack,
                       unsigned int *ticket, int sm_count, bool i16_out, const float *d_w_short = nullptr, int ls = 0, int step = 1)
{
    const uint32_t want = (n_groups + kLongWarps - 1) / kLongWarps;
    const uint32_t grid = want < (uint32_t)sm_count ? want : (uint32_t)sm_count;
    switch (step) {
#define LWB_LONG_CASE(CS)                                                                                                          \
    case CS:                                                                                                                       \
        if (i16_out) k_long<int16_t, CS><<<grid, kLongWarps * 32, kLongSmemBytes, stream>>>(d_runs, n_groups, d_pack, ticket, d_w_short, ls); \
        else k_long<float, CS><<<grid, kLongWarps * 32, kLongSmemBytes, stream>>>(d_runs, n_groups, d_pack, ticket, d_w_short, ls);          \
        break;
        LWB_LONG_STEPS(LWB_LONG_CASE)
#undef LWB_LONG_CASE
    default:
        return 1;
    }
    return cudaGetLastError() != cudaSuccess;
}
#endif  // __CUDACC__

}  // namespace lwb
