"""Interleaved PCM (LWB_OUT_F32_INTERLEAVED / LWB_OUT_I16_INTERLEAVED) on the fused long-block kernel (k_long): the
uniform-long device-memory batches that take k_long when planar take it when interleaved too (host-memory interleaved
batches keep the chain kernel, whose single pass measured faster than the sliced pipeline).  Every case is checked
against the
oracle (f32 bit-exact modulo the sign of zero, i16 exact) and byte for byte against the chain kernel, which writes
interleaved batches when LWB_NO_ITL=1: PCM, per-chain results and stream states."""
import contextlib
import os

import numpy as np
import pytest

import lewton_b200 as L
import vorbis_packer as vp
from helpers import RefStream, bits_equal, make_setup, mismatch_report, random_floor1_y
from lewton_b200 import _cabi as cabi
from lewton_b200 import frontend as fe
from test_frontend_gpu import consistent_modes, oracle_pcm

pytestmark = pytest.mark.gpu

N2 = 1024
SENTINEL_F32 = np.float32(-12345.5)
SENTINEL_I16 = np.int16(-31111)


@pytest.fixture(scope="module")
def ctx():
    c = L.Context(0)
    yield c
    c.close()


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: v for k, v in kv.items() if v is not None})
    for k, v in kv.items():
        if v is None:
            os.environ.pop(k, None)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def fmt_of(i16):
    return cabi.OUT_I16_INTERLEAVED if i16 else cabi.OUT_F32_INTERLEAVED


def blank(n, i16):
    return np.full(n, SENTINEL_I16 if i16 else SENTINEL_F32, np.int16 if i16 else np.float32)


def run(ctx, chains, entry, memory, coeffs, pcm, fmt, **kw):
    """One lwb_decode_chains call; host arrays in and out whatever the memory space.  Returns (pcm, (launches, launches of
    k_long)): the second count tells the fused path from the chain kernel."""
    pcm = pcm.copy()
    l0, k0 = ctx.launch_count, ctx.long_launch_count
    if memory == cabi.MEM_HOST:
        L.decode_chains(ctx, chains, entry, memory, coeffs, pcm, fmt, **kw)
    else:
        d_in, d_out = ctx.device_alloc(coeffs.nbytes), ctx.device_alloc(pcm.nbytes)
        try:
            ctx.h2d(d_in, coeffs)
            ctx.h2d(d_out, pcm)
            L.decode_chains(ctx, chains, entry, memory, d_in, d_out, fmt, **kw)
            ctx.synchronize()
            ctx.d2h(pcm, d_out)
        finally:
            ctx.device_free(d_in)
            ctx.device_free(d_out)
    return pcm, (ctx.launch_count - l0, ctx.long_launch_count - k0)


def results(chains):
    return [(c.status, c.n_samples, c.packets_done) for c in chains]


def check_oracle(pcm, chains, want, C, i16, oracle):
    """want[s]: [C][n] f32 from the oracle; chain s wrote n frames at out_offset."""
    for s, c in enumerate(chains):
        n = want[s].shape[1]
        assert c.status == 0 and c.n_samples == n, (s, c.status, c.n_samples, n)
        got = pcm[c.out_offset: c.out_offset + n * C].reshape(n, C).T
        if i16:
            assert np.array_equal(got, oracle.quantise_i16(want[s])), s
        else:
            assert bits_equal(got, want[s]), (s, mismatch_report(got, want[s]))


def check_untouched(pcm, chains, C, i16):
    """Nothing outside each chain's [out_offset, out_offset + n_samples * C) was written."""
    mask = np.ones(pcm.size, bool)
    for c in chains:
        mask[c.out_offset: c.out_offset + c.n_samples * C] = False
    s = SENTINEL_I16 if i16 else SENTINEL_F32
    assert np.all(pcm[mask] == s), np.nonzero(pcm[mask] != s)[0][:8]


def layout(n_frames, C, gap):
    """out_offset of each chain: chain s gets n_frames[s] * C elements, `gap` elements apart (gap % 4 == 0)."""
    offs, o = [], gap
    for n in n_frames:
        offs.append(o)
        o += n * C + gap
    return offs, o


def spectrum_case(ctx, oracle, C, i16, memory, seed, S=4, P=37, gap=None):
    """Three consecutive spectrum-entry batches of S streams x P long blocks (few chains: every chain is cut into runs with
    primer packets), half the streams starting from an imported state; fused vs LWB_NO_ITL=1 vs oracle."""
    rng = np.random.default_rng(seed)
    su = make_setup(ctx, C, 8, 11)
    gap = (12 if memory == cabi.MEM_DEVICE else 0) if gap is None else gap
    init = [rng.standard_normal((C, N2)).astype(np.float32) * 0.1 if s % 2 else None for s in range(S)]
    side = {}
    for name, e in (("fused", None), ("chain", "1")):
        pw = [L.PreviousWindowRight(su) for _ in range(S)]
        ref = [oracle.Pwr(C, 11) for _ in range(S)]
        for s in range(S):
            if init[s] is not None:
                pw[s].set_data(init[s])
                ref[s].set_data(init[s])
        side[name] = (pw, ref, [])
    for batch in range(3):
        spec = (rng.standard_normal((S, P, C, N2)) * 0.3).astype(np.float32)
        if i16 and batch == 1:
            spec[0, min(3, P - 1)] *= 1e5          # far out of range: the clamp
        outs = {}
        for name, e in (("fused", None), ("chain", "1")):
            pw, ref, _ = side[name]
            nf = [P - (0 if not pw[s].is_empty() else 1) for s in range(S)]
            offs, total = layout([n * N2 for n in nf], C, gap)
            chains = [L.ChainSpec(pw[s], np.ones(P, np.uint8), coeff_offset=s * P * C * N2, out_offset=offs[s]) for s in range(S)]
            with env(LWB_NO_ITL=e):
                pcm, launches = run(ctx, chains, cabi.ENTRY_SPECTRUM, memory, spec, blank(total, i16), fmt_of(i16))
            want = []
            for s in range(S):
                parts = []
                for p in range(P):
                    rc, o = oracle.synth_spectrum(8, 11, 1, 1, 1, spec[s, p], ref[s])
                    assert rc == 0
                    parts.append(o)
                want.append(np.concatenate(parts, axis=1))
            check_oracle(pcm, chains, want, C, i16, oracle)
            if memory == cabi.MEM_DEVICE:
                check_untouched(pcm, chains, C, i16)
            for s in range(S):
                assert bits_equal(pw[s].data(), ref[s].data()), (name, batch, s)
            outs[name] = (pcm, results(chains), [p.data() for p in pw], launches)
        assert np.array_equal(outs["fused"][0].view(np.uint8), outs["chain"][0].view(np.uint8)), batch
        assert outs["fused"][1] == outs["chain"][1]
        assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(outs["fused"][2], outs["chain"][2]))
        # device memory: k_long alone; host memory: the chain kernel, as with LWB_NO_ITL=1
        fused_long = 1 if memory == cabi.MEM_DEVICE else 0
        assert outs["fused"][3][1] == fused_long and outs["chain"][3][1] == 0, (outs["fused"][3], outs["chain"][3])
        if memory == cabi.MEM_DEVICE:
            assert outs["fused"][3][0] == 1, outs["fused"][3]
    return su


@pytest.mark.parametrize("C", [1, 2, 3, 6, 8])
@pytest.mark.parametrize("i16", [False, True])
@pytest.mark.parametrize("memory", [cabi.MEM_DEVICE, cabi.MEM_HOST])
def test_spectrum_entry_uniform_long(ctx, oracle, C, i16, memory):
    spectrum_case(ctx, oracle, C, i16, memory, seed=600 + 10 * C + 2 * int(i16) + int(memory == cabi.MEM_HOST))


@pytest.mark.parametrize("C,i16", [(2, False), (6, True)])
def test_spectrum_entry_many_chains_not_cut(ctx, oracle, C, i16):
    """Enough chains to fill the machine (no cuts), small gaps between them."""
    spectrum_case(ctx, oracle, C, i16, cabi.MEM_DEVICE, seed=650 + C, S=700, P=3, gap=4)


@pytest.mark.parametrize("i16", [False, True])
def test_interleaved_equals_planar_transposed(ctx, oracle, i16):
    """The fused interleaved output is the fused planar output, frame-major."""
    rng = np.random.default_rng(660 + int(i16))
    S, P, C = 64, 9, 2
    su = make_setup(ctx, C, 8, 11)
    spec = (rng.standard_normal((S, P, C, N2)) * 0.3).astype(np.float32)
    n = (P - 1) * N2
    planar = [L.ChainSpec(L.PreviousWindowRight(su), np.ones(P, np.uint8), coeff_offset=s * P * C * N2,
                          out_offset=s * C * n, out_stride=n) for s in range(S)]
    itl = [L.ChainSpec(L.PreviousWindowRight(su), np.ones(P, np.uint8), coeff_offset=s * P * C * N2,
                       out_offset=s * C * n) for s in range(S)]
    pf = cabi.OUT_I16_PLANAR if i16 else cabi.OUT_F32_PLANAR
    a, _ = run(ctx, planar, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, spec, blank(S * C * n, i16), pf)
    b, launches = run(ctx, itl, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, spec, blank(S * C * n, i16), fmt_of(i16))
    assert launches == (1, 1)
    assert np.array_equal(a.reshape(S, C, n).transpose(0, 2, 1).ravel().view(np.uint8), b.view(np.uint8))
    assert all(np.array_equal(x.pwr.data().view(np.uint32), y.pwr.data().view(np.uint32)) for x, y in zip(planar, itl))


def test_batches_k_long_does_not_take(ctx, oracle):
    """Interleaved batches k_long does not take stay what they were: an out_offset that is not a multiple of 4, two
    channel counts in one batch, a bad mode number, an OLA-guard error mid-chain -- each byte-equal to LWB_NO_ITL=1
    (PCM, per-chain results, stream states), the all-long ones also equal to the oracle."""
    rng = np.random.default_rng(670)
    s2, s3 = make_setup(ctx, 2, 8, 11), make_setup(ctx, 3, 8, 11)
    long6 = np.ones(6, np.uint8)
    cases = {
        "unaligned": [(s2, long6, 2)],
        "two_counts": [(s2, long6, 0), (s3, long6, 20000)],
        "bad_mode": [(s2, long6, 0), (s2, np.array([1, 1, 7, 1, 1, 1], np.uint8), 20000)],
        "ola_guard": [(s2, np.array([1, 1, 0, 1, 1, 1], np.uint8), 0), (s2, long6, 20000)],
    }

    def n_coeffs(su, modes):
        return su.audio_channels * sum(128 if m == 0 else N2 for m in modes)

    for name, streams in cases.items():
        spec = (rng.standard_normal(sum(n_coeffs(su, m) for su, m, _ in streams)) * 0.2).astype(np.float32)
        outs = {}
        for e in (None, "1"):
            pws, chains, co = [], [], 0
            for su, modes, o in streams:
                pws.append(L.PreviousWindowRight(su))
                chains.append(L.ChainSpec(pws[-1], modes, coeff_offset=co, out_offset=o))
                co += n_coeffs(su, modes)
            with env(LWB_NO_ITL=e):
                pcm, _ = run(ctx, chains, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, spec, blank(50000, False), cabi.OUT_F32_INTERLEAVED)
            outs[e] = (pcm, results(chains), [None if p.is_empty() else p.data() for p in pws])
        a, b = outs[None], outs["1"]
        assert np.array_equal(a[0].view(np.uint8), b[0].view(np.uint8)), name
        assert a[1] == b[1], (name, a[1], b[1])
        assert all((x is None) == (y is None) and (x is None or np.array_equal(x.view(np.uint32), y.view(np.uint32)))
                   for x, y in zip(a[2], b[2])), name
        if name == "bad_mode":
            assert a[1][0][0] == 0 and a[1][1][0] != 0, a[1]
        elif name == "ola_guard":
            assert a[1][0][0] == cabi.ERR_BAD_FORMAT and a[1][0][2] == 2 and a[1][1][0] == 0, a[1]
        else:
            co = 0
            for (su, modes, o), r in zip(streams, a[1]):
                Cn = su.audio_channels
                ref = oracle.Pwr(Cn, 11)
                parts = []
                for p in range(len(modes)):
                    x = spec[co + p * Cn * N2: co + (p + 1) * Cn * N2].reshape(Cn, N2)
                    rc, w = oracle.synth_spectrum(8, 11, 1, 1, 1, x, ref)
                    assert rc == 0
                    parts.append(w)
                co += n_coeffs(su, modes)
                w = np.concatenate(parts, axis=1)
                assert r[0] == 0 and r[1] == w.shape[1], (name, r)
                assert bits_equal(a[0][o: o + w.shape[1] * Cn].reshape(-1, Cn).T, w), name


def residue_batch(rng, refs, S, P, C, floors, mappings):
    res = (rng.standard_normal((S, P, C, N2)) * rng.integers(0, 2, (S, P, C, N2))).astype(np.float32)
    kinds = np.zeros((S, P, C), np.uint8)
    ys = np.zeros((S, P, C, cabi.MAX_POSTS), np.uint32)
    want = []
    for s in range(S):
        parts = []
        for p in range(P):
            fl = []
            for c in range(C):
                mult, xs = floors[mappings[0]["floor_of_channel"][c]]
                fl.append(None if rng.random() < 0.1 else random_floor1_y(rng, mult, len(xs)))
            k, y, _ = L.DecodedPacket(1, res[s, p], fl).pack()
            kinds[s, p], ys[s, p] = k, y
            if refs is not None:
                rc, o = refs[s].packet(1, 1, 1, res[s, p], fl)
                assert rc == 0
                parts.append(o)
        if refs is not None:
            want.append(np.concatenate(parts, axis=1))
    return res, kinds, ys, want


@pytest.mark.parametrize("C,i16,memory,chunks", [(2, False, cabi.MEM_DEVICE, None), (2, True, cabi.MEM_HOST, None),
                                                 (6, True, cabi.MEM_DEVICE, None), (6, False, cabi.MEM_HOST, "3"),
                                                 (3, False, cabi.MEM_HOST, "2")])
def test_residue_entry_uniform_long(ctx, oracle, C, i16, memory, chunks):
    """Full packets (coupling + floor-1), three consecutive batches.  Device memory: front stages + k_long (3 launches) vs
    the chain kernel (1).  Host memory, also with the slice count forced: the chain kernel either way."""
    rng = np.random.default_rng(700 + C + 10 * int(i16))
    S, P = 5, 9
    floors = [(2, [0, 1024, 300, 700, 100, 900])]
    mappings = [{"coupling": [(0, 1)] if C >= 2 else [], "floor_of_channel": [0] * C}]
    modes = ((0, 0), (1, 0))
    su = make_setup(ctx, C, 8, 11, modes=modes, mappings=mappings, floors=floors)
    sides = {}
    for name in ("fused", "chain"):
        sides[name] = ([L.PreviousWindowRight(su) for _ in range(S)], [RefStream(oracle, C, 8, 11, modes, mappings, floors) for _ in range(S)])
    for batch in range(3):
        bstate = rng.bit_generator.state
        outs = {}
        for name, e in (("fused", None), ("chain", "1")):
            pw, refs = sides[name]
            rng.bit_generator.state = bstate
            res, kinds, ys, want = residue_batch(rng, refs, S, P, C, floors, mappings)
            nf = [w.shape[1] for w in want]
            offs, total = layout(nf, C, 0)
            chains = [L.ChainSpec(pw[s], np.ones(P, np.uint8), coeff_offset=s * P * C * N2, packet_index=s * P, out_offset=offs[s])
                      for s in range(S)]
            with env(LWB_NO_ITL=e, LWB_E2E_CHUNKS=chunks):
                pcm, launches = run(ctx, chains, cabi.ENTRY_RESIDUE, memory, res, blank(total, i16), fmt_of(i16),
                                    floor_kind=kinds, floor1_y=ys)
            check_oracle(pcm, chains, want, C, i16, oracle)
            for s in range(S):
                assert bits_equal(pw[s].data(), refs[s].pwr.data()), (name, batch, s)
            outs[name] = (pcm, results(chains), [p.data() for p in pw], launches)
        assert np.array_equal(outs["fused"][0].view(np.uint8), outs["chain"][0].view(np.uint8)), batch
        assert outs["fused"][1] == outs["chain"][1]
        assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(outs["fused"][2], outs["chain"][2]))
        want_fused = (3, 1) if memory == cabi.MEM_DEVICE else (1, 0)
        assert outs["fused"][3] == want_fused and outs["chain"][3] == (1, 0), (outs["fused"][3], outs["chain"][3])


@pytest.mark.parametrize("i16", [False, True])
def test_prepared_plan_replays_and_replans(ctx, oracle, i16):
    """A plan created with an interleaved format: replayed (one k_long launch each), re-planned after a stream reset."""
    rng = np.random.default_rng(720 + int(i16))
    S, P, C = 6, 9, 3
    su = make_setup(ctx, C, 8, 11)
    pwrs = [L.PreviousWindowRight(su) for _ in range(S)]
    refs = [oracle.Pwr(C, 11) for _ in range(S)]
    spec = np.zeros((S, P, C, N2), np.float32)
    n = P * N2
    total = S * C * n
    dt = np.int16 if i16 else np.float32
    d_in, d_out = ctx.device_alloc(spec.nbytes), ctx.device_alloc(total * np.dtype(dt).itemsize)
    chains = [L.ChainSpec(pwrs[s], np.ones(P, np.uint8), coeff_offset=s * P * C * N2, out_offset=s * C * n) for s in range(S)]
    batch = L.Batch(ctx, chains, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, d_in, d_out, fmt_of(i16))
    try:
        for it in range(6):
            spec[:] = (rng.standard_normal(spec.shape) * 0.3).astype(np.float32)
            if it == 3:
                pwrs[2].reset()
                refs[2].reset()
            ctx.h2d(d_in, spec)
            ctx.h2d(d_out, blank(total, i16))
            l0, k0 = ctx.launch_count, ctx.long_launch_count
            batch.run()
            ctx.synchronize()
            assert (ctx.launch_count - l0, ctx.long_launch_count - k0) == (1, 1)
            pcm = np.empty(total, dt)
            ctx.d2h(pcm, d_out)
            batch.collect()
            want = []
            for s in range(S):
                parts = []
                for p in range(P):
                    rc, o = oracle.synth_spectrum(8, 11, 1, 1, 1, spec[s, p], refs[s])
                    assert rc == 0
                    parts.append(o)
                want.append(np.concatenate(parts, axis=1))
            check_oracle(pcm, chains, want, C, i16, oracle)
            check_untouched(pcm, chains, C, i16)
            for s in range(S):
                assert bits_equal(pwrs[s].data(), refs[s].data()), (it, s)
    finally:
        batch.close()
        ctx.device_free(d_in)
        ctx.device_free(d_out)


@pytest.mark.parametrize("entry", [cabi.ENTRY_RESIDUE, cabi.ENTRY_VQ])
def test_batcher_end_to_end_i16_interleaved(ctx, oracle, entry):
    """Real bitstreams (all long blocks) through lwf_batcher_decode with LWB_OUT_I16_INTERLEAVED: equal to the oracle
    and to LWB_NO_ITL=1.  The batcher's arenas are host memory, so k_long does not run."""
    rng = np.random.default_rng(740 + entry)
    C, P, S = 2, 10, 12
    spec = vp.StreamSpec(rng, channels=C)
    hdr = fe.Headers(spec.ident_packet(), spec.comment_packet(), spec.setup_packet())
    su = hdr.make_setup(ctx)
    distinct = []
    for d in range(3):
        pkts, infos = [], []
        for mode, prev, nxt in consistent_modes(spec, rng, P, p_short=0.0):
            pk, info = spec.audio_packet(mode, prev, nxt)
            pkts.append(pk)
            infos.append(info)
        distinct.append((pkts, np.concatenate(oracle_pcm(oracle, spec, infos)[0], axis=1)))
    stride = P * N2
    outs = {}
    for e in (None, "1"):
        pwrs = [L.PreviousWindowRight(su) for _ in range(S)]
        jobs = [(pwrs[s], list(distinct[s % 3][0])) for s in range(S)]
        pcm = np.full(S * C * stride, SENTINEL_I16, np.int16)
        bt = fe.StreamBatcher(ctx, hdr, threads=2, entry=entry)
        k0 = ctx.long_launch_count
        try:
            with env(LWB_NO_ITL=e):
                res = bt.decode(jobs, pcm, stride, out_format=cabi.OUT_I16_INTERLEAVED)
        finally:
            bt.close()
        assert ctx.long_launch_count == k0
        for s in range(S):
            w = distinct[s % 3][1]
            assert res[s] == (w.shape[1], P, 0), (e, s, res[s])
            got = pcm[s * C * stride: s * C * stride + w.shape[1] * C].reshape(-1, C).T
            assert np.array_equal(got, oracle.quantise_i16(w)), (e, s)
        outs[e] = (pcm, [p.data() for p in pwrs])
        for p in pwrs:
            p.close()
    for s in range(S):
        n = distinct[s % 3][1].shape[1]
        a = outs[None][0][s * C * stride: s * C * stride + n * C]
        b = outs["1"][0][s * C * stride: s * C * stride + n * C]
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), s
    assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(outs[None][1], outs["1"][1]))
