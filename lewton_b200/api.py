"""Host-side mirror of the reference's interface for the synthesis path, over the C ABI.

Names follow lewton (src/audio.rs, src/header.rs): `PreviousWindowRight`, `read_audio_packet`,
`read_audio_packet_generic`, `get_decoded_sample_count`, `FloorTypeOne`, `Mapping`, `ModeInfo`.
The one difference is where the packet enters: the reference function takes the raw packet bytes
and entropy-decodes them first (audio.rs:921-986, host/Rust work that stays where it is); here a
packet arrives as `DecodedPacket` = what that front half produces (mode, window flags, per-channel
floor Y values, dense residue vectors).  Everything after audio.rs:988 runs on the GPU.

This module is plumbing for tests, the bench and Python callers; the product is the shared
library.  It never computes audio on the CPU: without the library / a B200 it raises.
"""
import ctypes as C
import weakref

import numpy as np

from . import _cabi as cabi


class VorbisError(Exception):
    """lib.rs:119-125"""


class AudioReadError(VorbisError):
    """audio.rs:26-41; `.kind` is the variant name, `.code` the C status."""

    def __init__(self, code, detail=""):
        self.code = code
        self.kind = {cabi.ERR_BAD_FORMAT: "AudioBadFormat", cabi.ERR_BUFFER: "BufferNotAddressable",
                     cabi.ERR_MISMATCH: "Panic", cabi.ERR_INVALID: "InvalidArgument", cabi.ERR_CUDA: "Cuda",
                     cabi.ERR_NO_DEVICE: "NoDevice"}.get(code, f"Error{code}")
        super().__init__(f"{self.kind}{': ' + detail if detail else ''}")


def _ptr(a, typ=C.c_void_p):
    return a.ctypes.data_as(typ)


class Context:
    """One per GPU (lwb_ctx)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = cabi.lib().lwb_ctx_create(device, C.byref(self._h))
        if rc:
            self._h = None
            raise AudioReadError(rc, "lwb_ctx_create failed (no sm_100 device? there is no CPU fallback)")
        self.device = device
        self._children = weakref.WeakSet()      # setups / streams: destroyed before the ctx

    def check(self, rc):
        if rc:
            raise AudioReadError(rc, cabi.lib().lwb_last_error(self._h).decode())

    def synchronize(self):
        self.check(cabi.lib().lwb_ctx_synchronize(self._h))

    @property
    def cuda_stream(self):
        return cabi.lib().lwb_ctx_cuda_stream(self._h)

    @property
    def launch_count(self):
        return cabi.lib().lwb_ctx_launch_count(self._h)

    @property
    def long_launch_count(self):
        """Launches of the fused long-block kernels (k_long, k_long_s) among launch_count."""
        return cabi.lib().lwb_ctx_long_launch_count(self._h)

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self.check(cabi.lib().lwb_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, p):
        cabi.lib().lwb_device_free(self._h, p)

    def h2d(self, dst, arr):
        arr = np.ascontiguousarray(arr)
        self.check(cabi.lib().lwb_memcpy_h2d(self._h, dst, _ptr(arr), arr.nbytes))

    def d2h(self, arr, src):
        self.check(cabi.lib().lwb_memcpy_d2h(self._h, _ptr(arr), src, arr.nbytes))

    def close(self):
        if self._h:
            # readers (frontend.OggStreamReader) own streams and setups of their own: they go first
            for ch in [c for c in list(self._children) if not isinstance(c, (Batch, PreviousWindowRight, Setup))]:
                ch.close()
            for kind in (Batch, PreviousWindowRight, Setup):   # plans first, then streams, then setups
                for ch in [c for c in list(self._children) if isinstance(c, kind)]:
                    ch.close()
            cabi.lib().lwb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def generate_tables(bs):
    """CachedBlocksizeDerived::from_blocksize (header_cached.rs:33-41) via the library's host code."""
    if not 6 <= bs <= 13:
        raise AudioReadError(cabi.ERR_INVALID, "blocksize out of range")
    n = 1 << bs
    a, b = np.zeros(n // 2, np.float32), np.zeros(n // 2, np.float32)
    c, w = np.zeros(n // 4, np.float32), np.zeros(n // 2, np.float32)
    br = np.zeros(n // 8, np.uint32)
    rc = cabi.lib().lwb_tables_generate(bs, _ptr(a), _ptr(b), _ptr(c), _ptr(w), _ptr(br))
    if rc:
        raise AudioReadError(rc, "blocksize out of range")
    return {"a": a, "b": b, "c": c, "window": w, "bitrev": br}


class FloorTypeOne:
    """header.rs:415-424 (fields the synthesis half reads)."""

    def __init__(self, floor1_multiplier, floor1_x_list):
        self.floor1_multiplier = int(floor1_multiplier)
        self.floor1_x_list = [int(x) for x in floor1_x_list]


class FloorTypeZero:
    """header.rs:405-412: its curve is computed by the host and passed dense."""


class Mapping:
    """header.rs:384-390"""

    def __init__(self, channels, magnitudes=(), angles=(), mux=None, submap_floors=(0,)):
        self.mapping_magnitudes = list(magnitudes)
        self.mapping_angles = list(angles)
        self.mapping_mux = list(mux) if mux is not None else [0] * channels
        self.mapping_submap_floors = list(submap_floors)


class ModeInfo:
    """header.rs:393-396"""

    def __init__(self, mode_blockflag, mode_mapping=0):
        self.mode_blockflag = bool(mode_blockflag)
        self.mode_mapping = int(mode_mapping)


class Setup:
    """IdentHeader (header.rs:188-211) + the SetupHeader parts (header.rs:471-477) the path reads."""

    def __init__(self, ctx, audio_channels, blocksize_0, blocksize_1, floors, mappings, modes, tables=None):
        self.ctx = ctx
        self.audio_channels, self.blocksize_0, self.blocksize_1 = audio_channels, blocksize_0, blocksize_1
        self.floors, self.mappings, self.modes = list(floors), list(mappings), list(modes)
        d = cabi.SetupDesc()
        d.audio_channels, d.blocksize_0, d.blocksize_1 = audio_channels, blocksize_0, blocksize_1
        self._keep = []
        if tables is not None:          # [(dict for bs0), (dict for bs1)] like generate_tables()
            for i, t in enumerate(tables):
                arrs = {k: np.ascontiguousarray(t[k]) for k in ("a", "b", "c", "window", "bitrev")}
                self._keep.append(arrs)
                d.tables[i].a = _ptr(arrs["a"], cabi.fp)
                d.tables[i].b = _ptr(arrs["b"], cabi.fp)
                d.tables[i].c = _ptr(arrs["c"], cabi.fp)
                d.tables[i].window = _ptr(arrs["window"], cabi.fp)
                d.tables[i].bitrev = _ptr(arrs["bitrev"], cabi.u32p)
        fl = (cabi.FloorDesc * len(self.floors))()
        for i, f in enumerate(self.floors):
            if isinstance(f, FloorTypeOne):
                fl[i].floor_type = cabi.FLOOR_TYPE_ONE
                fl[i].floor1_multiplier = f.floor1_multiplier
                fl[i].floor1_values = len(f.floor1_x_list)
                for k, x in enumerate(f.floor1_x_list[: cabi.MAX_POSTS]):
                    fl[i].floor1_x_list[k] = x
            else:
                fl[i].floor_type = cabi.FLOOR_TYPE_ZERO
        mp = (cabi.MappingDesc * len(self.mappings))()
        for i, m in enumerate(self.mappings):
            mp[i].coupling_steps = len(m.mapping_magnitudes)
            mp[i].submaps = len(m.mapping_submap_floors)
            for k, (a, b) in enumerate(zip(m.mapping_magnitudes, m.mapping_angles)):
                mp[i].magnitudes[k], mp[i].angles[k] = a, b
            for k, v in enumerate(m.mapping_mux):
                mp[i].mux[k] = v
            for k, v in enumerate(m.mapping_submap_floors):
                mp[i].submap_floors[k] = v
        md = (cabi.ModeDesc * len(self.modes))()
        for i, m in enumerate(self.modes):
            md[i].blockflag, md[i].mapping = int(m.mode_blockflag), m.mode_mapping
        d.n_floors, d.floors = len(self.floors), fl
        d.n_mappings, d.mappings = len(self.mappings), mp
        d.n_modes, d.modes = len(self.modes), md
        self._h = C.c_void_p()
        rc = cabi.lib().lwb_setup_create(ctx._h, C.byref(d), C.byref(self._h))
        if rc:
            self._h = None
            raise AudioReadError(rc, cabi.lib().lwb_last_error(ctx._h).decode())
        ctx._children.add(self)

    @classmethod
    def _adopt(cls, ctx, handle, audio_channels, blocksize_0, blocksize_1, mode_blockflags=()):
        """Wrap an lwb_setup built by the library itself (lwf_headers_make_setup)."""
        self = cls.__new__(cls)
        self.ctx = ctx
        self.audio_channels, self.blocksize_0, self.blocksize_1 = audio_channels, blocksize_0, blocksize_1
        self.floors, self.mappings = [], []
        self.modes = [ModeInfo(bool(b)) for b in mode_blockflags]
        self._keep = []
        self._h = C.c_void_p(handle)
        ctx._children.add(self)
        return self

    def blocksize(self, mode_number):
        if not 0 <= mode_number < len(self.modes):
            raise AudioReadError(cabi.ERR_BAD_FORMAT, "mode number out of range (audio.rs:926-930)")
        return 1 << (self.blocksize_1 if self.modes[mode_number].mode_blockflag else self.blocksize_0)

    def close(self):
        if self._h:
            if self.ctx._h:
                cabi.lib().lwb_setup_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PreviousWindowRight:
    """audio.rs:847-861 -- the only inter-packet state, resident on the device (lwb_stream)."""

    def __init__(self, setup, _handle=None):
        self.setup = setup
        self._h = _handle or C.c_void_p()
        if _handle is None:
            setup.ctx.check(cabi.lib().lwb_stream_open(setup.ctx._h, setup._h, C.byref(self._h)))
        setup.ctx._children.add(self)

    @classmethod
    def new(cls, setup):
        return cls(setup)

    def is_empty(self):
        return bool(cabi.lib().lwb_stream_is_empty(self._h))

    def reset(self):
        cabi.lib().lwb_stream_reset(self._h)

    def clone(self):
        h = C.c_void_p()
        self.setup.ctx.check(cabi.lib().lwb_stream_clone(self._h, C.byref(h)))
        return PreviousWindowRight(self.setup, h)

    def __len__(self):
        return cabi.lib().lwb_stream_state_len(self._h)

    def data(self):
        if self.is_empty():
            return None
        out = np.zeros((self.setup.audio_channels, len(self)), np.float32)
        self.setup.ctx.check(cabi.lib().lwb_stream_export_state(self._h, _ptr(out)))
        return out

    def set_data(self, arr):
        arr = np.ascontiguousarray(arr, np.float32)
        assert arr.shape[0] == self.setup.audio_channels
        self.setup.ctx.check(cabi.lib().lwb_stream_import_state(self._h, _ptr(arr), arr.shape[1]))

    def close(self):
        if self._h:
            if self.setup.ctx._h:
                cabi.lib().lwb_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DecodedPacket:
    """What audio.rs:921-986 hands to the synthesis half.

    floors: per channel  None (DecodedFloor::Unused) | sequence of floor1 Y values
            (DecodedFloor::TypeOne) | float32 ndarray of n/2 (a floor-0 curve computed by the host)
    residue: [channels][n/2] float32
    """

    def __init__(self, mode_number, residue, floors, prev_window_flag=True, next_window_flag=True):
        self.mode_number = mode_number
        self.prev_window_flag, self.next_window_flag = bool(prev_window_flag), bool(next_window_flag)
        self.residue = np.ascontiguousarray(residue, np.float32)
        self.floors = list(floors)

    def pack(self):
        ch, n2 = self.residue.shape
        kinds = np.zeros(ch, np.uint8)
        ys = np.zeros((ch, cabi.MAX_POSTS), np.uint32)
        dense = None
        for c, f in enumerate(self.floors):
            if f is None:
                kinds[c] = cabi.FLOOR_UNUSED
            elif isinstance(f, np.ndarray) and f.dtype.kind == "f":
                kinds[c] = cabi.FLOOR_DENSE
                if dense is None:
                    dense = np.zeros((ch, n2), np.float32)
                dense[c] = f
            else:
                kinds[c] = cabi.FLOOR_ONE
                ys[c, : len(f)] = np.asarray(f, np.uint32)
        return kinds, ys, dense


_FORMATS = {("f32", False): (cabi.OUT_F32_PLANAR, np.float32), ("i16", False): (cabi.OUT_I16_PLANAR, np.int16),
            ("f32", True): (cabi.OUT_F32_INTERLEAVED, np.float32), ("i16", True): (cabi.OUT_I16_INTERLEAVED, np.int16)}


def get_decoded_sample_count(setup, mode_number, prev_window_flag=True, next_window_flag=True):
    """audio.rs:874-909 for an already parsed packet header."""
    n = C.c_uint32()
    rc = cabi.lib().lwb_decoded_sample_count(setup._h, mode_number, int(prev_window_flag), int(next_window_flag),
                                             C.byref(n))
    if rc:
        raise AudioReadError(rc)
    return n.value


def read_audio_packet_generic(setup, packet, pwr, sample="f32", interleaved=False):
    """audio.rs:919-1160 (back half).  Returns planar [channels][len] (Vec<Vec<S>>) or
    interleaved [len][channels] (InterleavedSamples<S>); len == 0 for the first packet after a reset.
    Raises AudioReadError (kind 'AudioBadFormat' for the guard at audio.rs:1107-1111)."""
    fmt, dt = _FORMATS[(sample, interleaved)]
    ch = setup.audio_channels
    cap = setup.blocksize(packet.mode_number)
    kinds, ys, dense = packet.pack()
    p = cabi.Packet()
    p.mode_number = packet.mode_number
    p.prev_window_flag, p.next_window_flag = int(packet.prev_window_flag), int(packet.next_window_flag)
    p.floor_kind = _ptr(kinds, cabi.u8p)
    p.floor1_y = _ptr(ys, cabi.u32p)
    if dense is not None:
        p.dense_floor = _ptr(dense, cabi.fp)
    p.residue = _ptr(packet.residue, cabi.fp)
    out = np.zeros((cap, ch) if interleaved else (ch, cap), dt)
    n = C.c_size_t()
    rc = cabi.lib().lwb_decode_packet(pwr._h, C.byref(p), fmt, _ptr(out), cap, C.byref(n))
    if rc:
        raise AudioReadError(rc, cabi.lib().lwb_last_error(setup.ctx._h).decode())
    return out[: n.value].copy() if interleaved else out[:, : n.value].copy()


def read_audio_packet(setup, packet, pwr):
    """audio.rs:1170-1173: Vec<Vec<i16>>."""
    return read_audio_packet_generic(setup, packet, pwr, sample="i16", interleaved=False)


def decode_spectrum(setup, mode_number, spectrum, pwr, prev_window_flag=True, next_window_flag=True, sample="f32",
                    interleaved=False):
    """Entry at the record_pre_mdct tap (audio.rs:1041): spectrum [channels][n/2] = floor x residue."""
    fmt, dt = _FORMATS[(sample, interleaved)]
    ch = setup.audio_channels
    cap = setup.blocksize(mode_number)
    sp = np.ascontiguousarray(spectrum, np.float32)
    out = np.zeros((cap, ch) if interleaved else (ch, cap), dt)
    n = C.c_size_t()
    rc = cabi.lib().lwb_decode_spectrum(pwr._h, mode_number, int(prev_window_flag), int(next_window_flag), _ptr(sp), fmt,
                                        _ptr(out), cap, C.byref(n))
    if rc:
        raise AudioReadError(rc, cabi.lib().lwb_last_error(setup.ctx._h).decode())
    return out[: n.value].copy() if interleaved else out[:, : n.value].copy()


def debug_taps(setup, packet, pwr):
    """The reference's record_* taps (lib.rs:56-94): post-inverse-coupling residue, pre-MDCT
    spectrum, post-MDCT samples.  Does not modify the state."""
    ch = setup.audio_channels
    n = setup.blocksize(packet.mode_number)
    kinds, ys, dense = packet.pack()
    p = cabi.Packet()
    p.mode_number = packet.mode_number
    p.prev_window_flag, p.next_window_flag = int(packet.prev_window_flag), int(packet.next_window_flag)
    p.floor_kind, p.floor1_y = _ptr(kinds, cabi.u8p), _ptr(ys, cabi.u32p)
    if dense is not None:
        p.dense_floor = _ptr(dense, cabi.fp)
    p.residue = _ptr(packet.residue, cabi.fp)
    a, b, c = (np.zeros((ch, n // 2), np.float32), np.zeros((ch, n // 2), np.float32), np.zeros((ch, n), np.float32))
    setup.ctx.check(cabi.lib().lwb_debug_packet_taps(pwr._h, C.byref(p), _ptr(a), _ptr(b), _ptr(c)))
    return a, b, c


class ChainSpec:
    """One stream's run of consecutive packets inside a batch (lwb_chain)."""

    def __init__(self, pwr, mode_numbers, prev_flags=None, next_flags=None, coeff_offset=0, packet_index=0,
                 out_offset=0, out_stride=0):
        self.pwr = pwr
        self.modes = np.ascontiguousarray(mode_numbers, np.uint8)
        self.prev = None if prev_flags is None else np.ascontiguousarray(prev_flags, np.uint8)
        self.next = None if next_flags is None else np.ascontiguousarray(next_flags, np.uint8)
        self.coeff_offset, self.packet_index = coeff_offset, packet_index
        self.out_offset, self.out_stride = out_offset, out_stride
        self.n_samples = self.packets_done = self.status = 0


class Batch:
    """A prepared lwb_decode_chains call: the lwb_chain array and lwb_batch_io are built once, so a
    hot loop pays only the C call (the per-step Python cost of marshalling thousands of chains
    would otherwise exceed the kernel time)."""

    def __init__(self, ctx, chains, entry, memory, coeffs, pcm, out_format, floor_kind=None, floor1_y=None,
                 dense_floor=None, floor_memory=cabi.MEM_HOST, vq=None):
        """vq: LWB_ENTRY_VQ arrays (runs, run_offsets, entries, entry_offsets): numpy arrays or device pointers."""
        self.ctx, self.chains = ctx, list(chains)
        self._keep = (coeffs, pcm, floor_kind, floor1_y, dense_floor, vq)
        self._arr = arr = (cabi.Chain * len(self.chains))()
        for i, c in enumerate(self.chains):
            arr[i].stream = c.pwr._h
            arr[i].n_packets = len(c.modes)
            arr[i].mode_numbers = _ptr(c.modes, cabi.u8p)
            if c.prev is not None:
                arr[i].prev_window_flags = _ptr(c.prev, cabi.u8p)
            if c.next is not None:
                arr[i].next_window_flags = _ptr(c.next, cabi.u8p)
            arr[i].coeff_offset, arr[i].packet_index = c.coeff_offset, c.packet_index
            arr[i].out_offset, arr[i].out_stride = c.out_offset, c.out_stride

        def addr(x):
            if x is None:
                return None
            if isinstance(x, np.ndarray):
                return x.ctypes.data
            return int(x)

        self._io = io = cabi.BatchIo()
        io.entry, io.memory, io.out_format = entry, memory, out_format
        io.coeffs, io.pcm, io.dense_floor = addr(coeffs), addr(pcm), addr(dense_floor)
        io.floor_kind, io.floor1_y = addr(floor_kind), addr(floor1_y)
        io.floor_memory = floor_memory
        if vq is not None:
            io.vq_runs, io.vq_run_offsets, io.vq_entries, io.vq_entry_offsets = (addr(x) for x in vq)
        self._n = len(self.chains)
        self._plan = C.c_void_p()
        ctx.check(cabi.lib().lwb_plan_create(ctx._h, self._arr, self._n, C.byref(self._io), C.byref(self._plan)))
        ctx._children.add(self)
        self._fn = cabi.lib().lwb_plan_execute

    def run(self):
        """One submission (lwb_plan_execute).  Results land in the chain array; collect() copies them back."""
        rc = self._fn(self._plan)
        if rc:
            self.ctx.check(rc)

    def close(self):
        if self._plan:
            if self.ctx._h:
                cabi.lib().lwb_plan_destroy(self._plan)
            self._plan = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def collect(self):
        for i, c in enumerate(self.chains):
            c.n_samples, c.packets_done, c.status = self._arr[i].n_samples, self._arr[i].packets_done, self._arr[i].status
        return self.chains


def decode_chains(ctx, chains, entry, memory, coeffs, pcm, out_format, floor_kind=None, floor1_y=None,
                  dense_floor=None, floor_memory=cabi.MEM_HOST, vq=None):
    """lwb_decode_chains.  coeffs/pcm/dense_floor: numpy arrays (MEM_HOST) or integer device
    pointers (MEM_DEVICE); floor_kind/floor1_y: numpy arrays (floor_memory MEM_HOST) or integer
    device pointers (MEM_DEVICE)."""
    b = Batch(ctx, chains, entry, memory, coeffs, pcm, out_format, floor_kind, floor1_y, dense_floor, floor_memory, vq)
    try:
        b.run()
        return b.collect()
    finally:
        b.close()
