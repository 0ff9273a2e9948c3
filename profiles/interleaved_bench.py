#!/usr/bin/env python3
"""Interleaved PCM against planar PCM on the fused kernels.  For each workload and output format it times, in the same
process and alternating round by round:

  planar_fused   the planar format (the fused kernel's home ground);
  itl_fused      the interleaved format as dispatched by default;
  itl_chain      the interleaved format with LWB_NO_ITL=1 (the chain kernel, what interleaved batches ran on before).

Device-resident buffers (working sets above the 126 MB L2), prepared batches (lwb_plan_execute), state carried from
step to step, CUDA events around `IB_REPS` steps after two warm-up steps.  Algorithmic bytes are those of planar output:
8 B per sample for f32 (4 in, 4 out), 6 B for i16.  At the timed size, after the last step, the itl_fused output must
equal the itl_chain output and the planar output transposed, byte for byte (the script fails otherwise).

The host-memory workload (residue entry, i16 interleaved, every host array pinned) is timed with a host clock around
lwb_decode_chains, which synchronises.  One JSON line per (workload, format, path), with the card name and power limit
read in the same run.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PATHS = ("planar_fused", "itl_fused", "itl_chain")


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def set_itl_env(path):
    if path == "itl_chain":
        os.environ["LWB_NO_ITL"] = "1"
    else:
        os.environ.pop("LWB_NO_ITL", None)


def long_workload(L, cabi, ctx, torch, C, S, P, residue):
    """S streams x P long blocks of C channels: spectrum entry, or the residue entry with floor-1 on every channel."""
    from helpers import random_floor1_y
    modes = [L.ModeInfo(False), L.ModeInfo(True)]
    floors = [L.FloorTypeOne(2, [0, 1024, 300, 700, 100, 900, 40, 500])]
    coupling = ([0], [1]) if residue and C >= 2 else ((), ())
    su = L.Setup(ctx, C, 8, 11, floors, [L.Mapping(C, coupling[0], coupling[1])], modes)
    n_in = S * P * C * 1024
    coeffs = torch.randn(n_in, device="cuda") * 3e-2
    kw = {}
    if residue:
        rng = np.random.default_rng(5)
        res1 = np.zeros((C, 1024), np.float32)
        fl = [random_floor1_y(rng, 2, 8) for _ in range(C)]
        k, y, _ = L.DecodedPacket(1, res1, fl).pack()
        kinds = np.ascontiguousarray(np.broadcast_to(k, (S * P, C)))
        ys = np.ascontiguousarray(np.broadcast_to(y, (S * P,) + y.shape))
        kw = dict(floor_kind=kinds, floor1_y=ys)
    return su, coeffs, kw


def run_device(L, cabi, ctx, torch, stream, name, C, S, P, residue, i16, reps, rounds, card_info):
    su, coeffs, kw = long_workload(L, cabi, ctx, torch, C, S, P, residue)
    entry = cabi.ENTRY_RESIDUE if residue else cabi.ENTRY_SPECTRUM
    dt = torch.int16 if i16 else torch.float32
    region = P * 1024
    fmts = {"planar_fused": cabi.OUT_I16_PLANAR if i16 else cabi.OUT_F32_PLANAR}
    fmts["itl_fused"] = fmts["itl_chain"] = cabi.OUT_I16_INTERLEAVED if i16 else cabi.OUT_F32_INTERLEAVED
    state = {}
    for path in PATHS:
        set_itl_env(path)
        pw = [L.PreviousWindowRight(su) for _ in range(S)]
        pcm = torch.zeros(S * C * region, dtype=dt, device="cuda")
        planar = path == "planar_fused"
        chains = [L.ChainSpec(pw[s], np.ones(P, np.uint8), coeff_offset=s * P * C * 1024, packet_index=s * P,
                              out_offset=s * C * region, out_stride=region if planar else 0) for s in range(S)]
        b = L.Batch(ctx, chains, entry, cabi.MEM_DEVICE, coeffs.data_ptr(), pcm.data_ptr(), fmts[path], **kw)
        l0 = ctx.launch_count
        b.run()
        ctx.synchronize()
        launches = ctx.launch_count - l0
        b.run()                                  # warm-up: steady state (every stream has history)
        ctx.synchronize()
        state[path] = dict(pw=pw, pcm=pcm, chains=chains, batch=b, launches=launches, ms=[])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for path in PATHS:
            set_itl_env(path)
            st = state[path]
            e0.record(stream)
            for _ in range(reps):
                st["batch"].run()
            e1.record(stream)
            ctx.synchronize()
            st["ms"].append(e0.elapsed_time(e1) / reps)
    os.environ.pop("LWB_NO_ITL", None)
    # byte equality after the same number of steps on every path
    a = state["itl_fused"]["pcm"]
    assert torch.equal(a, state["itl_chain"]["pcm"]), f"{name}: interleaved fused != LWB_NO_ITL=1"
    pt = state["planar_fused"]["pcm"].view(S, C, region).transpose(1, 2).reshape(-1)
    assert torch.equal(a, pt), f"{name}: interleaved fused != planar transposed"
    for path in PATHS:
        st = state[path]
        st["batch"].collect()
        samples = sum(c.n_samples for c in st["chains"]) * C
        ms = float(np.median(st["ms"]))
        gbs = samples * (6 if i16 else 8) / ms / 1e6
        print(json.dumps({"workload": name, "format": "i16" if i16 else "f32", "path": path, "channels": C, "streams": S,
                          "packets": P, "entry": "residue" if residue else "spectrum", "memory": "device",
                          "ms_median": ms, "ms_all": st["ms"], "launches_per_step": st["launches"],
                          "msamples_per_s": samples / ms / 1e3, "algorithmic_gbs": gbs, "frac_of_7700_gbs": gbs / 7700.0,
                          "card": card_info[0], "power_limit": card_info[1], "outputs_equal": True}), flush=True)
        st["batch"].close()
        for p in st["pw"]:
            p.close()
    su.close()
    del state, coeffs
    torch.cuda.empty_cache()


def run_host_e2e(L, cabi, ctx, torch, name, C, S, P, reps, rounds, card_info):
    """Residue entry, host memory (pinned), i16: the PCM comes home over PCIe in slices."""
    su, _, kw = long_workload(L, cabi, ctx, torch, C, 1, 1, True)
    rng = np.random.default_rng(9)
    kinds1, ys1 = kw["floor_kind"][0], kw["floor1_y"][0]
    # every host array pinned, as the batcher's arenas are: pageable copies would time the host's memcpy instead
    kinds = torch.empty((S * P, C), dtype=torch.uint8, pin_memory=True).numpy()
    kinds[:] = kinds1
    ys = torch.empty((S * P,) + ys1.shape, dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
    ys[:] = ys1
    res = torch.empty(S * P * C * 1024, dtype=torch.float32, pin_memory=True).numpy()
    res[:] = (rng.standard_normal(res.size) * 3e-2).astype(np.float32)
    region = P * 1024
    outs, times, launches = {}, {p: [] for p in PATHS}, {}
    pws = {p: [L.PreviousWindowRight(su) for _ in range(S)] for p in PATHS}
    pcms = {p: torch.zeros(S * C * region, dtype=torch.int16, pin_memory=True).numpy() for p in PATHS}

    def step(path):
        planar = path == "planar_fused"
        chains = [L.ChainSpec(pws[path][s], np.ones(P, np.uint8), coeff_offset=s * P * C * 1024, packet_index=s * P,
                              out_offset=s * C * region, out_stride=region if planar else 0) for s in range(S)]
        fmt = cabi.OUT_I16_PLANAR if planar else cabi.OUT_I16_INTERLEAVED
        L.decode_chains(ctx, chains, cabi.ENTRY_RESIDUE, cabi.MEM_HOST, res, pcms[path], fmt, floor_kind=kinds, floor1_y=ys)
        return chains

    for path in PATHS:
        set_itl_env(path)
        l0 = ctx.launch_count
        step(path)
        launches[path] = ctx.launch_count - l0
        step(path)
    for _ in range(rounds):
        for path in PATHS:
            set_itl_env(path)
            t0 = time.perf_counter()
            for _ in range(reps):
                chains = step(path)
            times[path].append((time.perf_counter() - t0) / reps * 1e3)
            outs[path] = chains
    os.environ.pop("LWB_NO_ITL", None)
    assert np.array_equal(pcms["itl_fused"], pcms["itl_chain"]), f"{name}: interleaved fused != LWB_NO_ITL=1"
    assert np.array_equal(pcms["itl_fused"], pcms["planar_fused"].reshape(S, C, region).transpose(0, 2, 1).ravel()), \
        f"{name}: interleaved fused != planar transposed"
    for path in PATHS:
        samples = sum(c.n_samples for c in outs[path]) * C
        ms = float(np.median(times[path]))
        print(json.dumps({"workload": name, "format": "i16", "path": path, "channels": C, "streams": S, "packets": P,
                          "entry": "residue", "memory": "host", "ms_median": ms, "ms_all": times[path],
                          "launches_per_call": launches[path], "msamples_per_s": samples / ms / 1e3,
                          "card": card_info[0], "power_limit": card_info[1], "outputs_equal": True}), flush=True)
        for p in pws[path]:
            p.close()
    su.close()


def main():
    import torch

    import lewton_b200 as L
    from lewton_b200 import _cabi as cabi

    card_info = card()
    reps, rounds = int(os.environ.get("IB_REPS", 40)), int(os.environ.get("IB_ROUNDS", 5))
    ctx = L.Context(0)
    stream = torch.cuda.ExternalStream(ctx.cuda_stream)
    only = os.environ.get("IB_ONLY")
    device_workloads = [
        ("headline_stereo_long", 2, 4096, 16, False),      # the bench.py shape
        ("six_channel_long", 6, 1024, 16, False),
        ("residue_entry_stereo_long", 2, 2048, 16, True),
    ]
    for name, C, S, P, residue in device_workloads:
        if only and name not in only.split(","):
            continue
        for i16 in (False, True):
            run_device(L, cabi, ctx, torch, stream, name, C, S, P, residue, i16, reps, rounds, card_info)
    if not only or "host_e2e_i16" in only.split(","):
        run_host_e2e(L, cabi, ctx, torch, "host_e2e_i16", 2, 2048, 16, max(1, reps // 2), rounds, card_info)
    ctx.close()


if __name__ == "__main__":
    main()
