#!/usr/bin/env python3
"""bench.py -- IMDCT + window + overlap-add throughput on synthetic 2048-sample long blocks.

Contract (see DESIGN.md "Measurement"):
  python bench.py --gpus N --steps K --warmup W          our arm (one process per GPU under torchrun)
  python bench.py --impl reference ...                   the CPU baseline arm (oracle port, host cores)

One step = one pass of the hot path over one batch: S independent stereo streams x P consecutive
long/long packets (spectrum [S][P][2][1024] f32, device-resident, > L2), through
lwb_decode_chains (fused kernel k_long).  `value` = channel-samples per second over all ranks,
timed with CUDA events on the library's stream, max over ranks.  `e2e` = the same call with HOST
(pinned) buffers: H2D of the spectrum and D2H of the PCM inside the timed region.

--dump-outputs DIR writes what the last timed step returned (inputs are seeded: the same arguments give the same
inputs), so that two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N2 = 1024
ALG_BYTES_PER_SAMPLE = 8          # 4 B spectrum read + 4 B f32 PCM write (SURVEY.md section 8d)
DUMP_PCM_BYTES = 48 << 20         # --dump-outputs: PCM sample size cap (the whole dump stays under 64 MB)
DUMP_SEED = 2024


def timed_outputs(pcm, batch):
    """--dump-outputs: what a caller of the timed step receives after its last run -- the PCM of a fixed, seeded
    sample of the streams (all of them when they fit DUMP_PCM_BYTES) and every chain's result fields."""
    S = pcm.shape[0]
    k = min(S, DUMP_PCM_BYTES // (pcm[0].numel() * pcm.element_size()))
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(S, k, replace=False))
    res = [(c.n_samples, c.packets_done, c.status) for c in batch.collect()]
    return {"pcm": pcm[idx.tolist()].cpu().numpy(),                   # [k][channels][packets * 1024] f32
            "pcm_streams": idx.astype(np.float64),                     # the sampled stream indices
            "chain_results": np.array(res, np.float64)}                # [streams][n_samples, packets_done, status]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(streams, packets):
    """DRAM bytes (read + write) per k_long launch from the committed `ncu --set full` capture of this
    same workload (profiles/*_k_long_ncu_summary.txt, newest round); None for any other workload."""
    if (streams, packets) != (4096, 16):
        return None, None
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_k_long_ncu_summary.txt")))
    if not files:
        return None, None
    txt = open(files[-1]).read()
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
        m = re.search(re.escape(key) + r"\s+([0-9.]+)\s+(\w+)", txt)
        if not m or m.group(2) not in unit:
            return None, None
        tot += float(m.group(1)) * unit[m.group(2)]
    return tot, os.path.relpath(files[-1], ROOT)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_threads():
    """Threads the CPU arm can really use: the smaller of the logical CPUs, this process's affinity
    mask and the container's CPU quota (cgroup v2 cpu.max)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def cpu_reference(streams, packets, threads, target_sec=2.0, seed=1234):
    """The oracle port (lewton-equivalent C restatement) on the host cores; returns
    (samples/s, seconds, reps).  The same synthetic input is swept `reps` times so that the timed
    region lasts about target_sec of wall clock on all `threads` cores."""
    from oracle import oracle
    oracle.build()
    rng = np.random.default_rng(seed)
    chains = streams * 2
    spec = (rng.standard_normal((chains, packets, N2)) * 1e-2).astype(np.float32)
    sec1, _ = oracle.bench_chains(11, spec, threads, 1)            # calibration pass (also warms caches)
    reps = max(1, int(target_sec / max(sec1, 1e-4)))
    sec, _ = oracle.bench_chains(11, spec, threads, reps)
    samples = chains * (packets - 1) * N2 * reps     # the first packet of a fresh chain emits nothing
    return samples / sec, sec, reps


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the crate is
    Rust and cannot be built here), all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = host_threads()
    streams, packets = 8 * threads, 17            # 16 chains per thread, swept ~0.5 s per step
    vals = []
    for i in range(args.warmup + args.steps):
        v, sec, reps = cpu_reference(streams, packets, threads, target_sec=0.5, seed=1234 + i)
        if i >= args.warmup:
            vals.append((v, sec))
    v = float(np.mean([a for a, _ in vals]))
    ms = float(np.mean([b for _, b in vals])) * 1e3
    line = {"impl": "reference", "metric": "Msamples/s IMDCT+window+OLA, 2048-pt long blocks", "value": v / 1e6,
            "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "stereo long-block (n=2048) packets, IMDCT+window+OLA, CPU oracle port",
                       "streams": streams, "packets_per_stream": packets, "channels": 2},
            "cpu_baseline": {"value": v / 1e6, "unit": "Msamples/s", "cores": threads, "kind": "port",
                             "sample": f"{streams} stereo streams x {packets} long packets swept ~0.5 s per step, "
                                       "lewton-equivalent C restatement (oracle/), the crate itself is Rust"},
            "e2e": {"value": v / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="stereo streams per GPU per step")
    ap.add_argument("--packets", type=int, default=16, help="consecutive long packets per stream per step")
    ap.add_argument("--e2e-streams", type=int, default=2048)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="leave the rank's CPU affinity / memory policy alone")
    ap.add_argument("--strong-streams", type=int, default=4096,
                    help="BASELINE.json configs[3]: this many stereo streams in TOTAL, sharded over the ranks (0 = skip)")
    ap.add_argument("--strong-packets", type=int, default=64)
    ap.add_argument("--mixed-streams", type=int, default=2048,
                    help="streams per GPU of the mixed short/long measurement (0: skip)")
    ap.add_argument("--sustained-sec", type=float, default=1.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's outputs of the last one as DIR/<name>.npy (pcm: a seeded "
                         "sample of the streams; pcm_streams: their indices; chain_results: per-chain n_samples, "
                         "packets_done, status)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path; the reference arm has no outputs to dump")
    if args.dump_outputs and 2 * args.packets * N2 * 4 > DUMP_PCM_BYTES:
        ap.error(f"--dump-outputs: one stream's PCM exceeds {DUMP_PCM_BYTES >> 20} MB; use fewer --packets")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import lewton_b200 as L
    from lewton_b200 import _cabi as cabi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line.  NCCL prints its banner / INFO lines to stdout: instead of silencing
    # NCCL_DEBUG (which hid the communicator's rank count from whoever launched us), file descriptor 1 is pointed
    # at stderr for the whole run and the JSON line is written to the saved descriptor at the end.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    # Host side of e2e: bind this rank to the CPUs / memory of the NUMA node its GPU hangs off BEFORE any pinned
    # allocation (first touch then lands on the local node); the original mask is restored for the CPU arm.
    affinity0 = os.sched_getaffinity(0)
    numa = cabi.lib().lwb_bind_host_to_device(local) if not args.no_numa_bind else -1
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(local)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"

    ctx = L.Context(local)
    # weak scaling: every rank owns `--streams` streams (global stream ids [lo, hi), contiguous ranges,
    # lewton_b200/sharding.py); no data-path collective
    from lewton_b200.sharding import stream_range
    lo, hi = stream_range(args.streams * world, world, rank)
    S, P, C = hi - lo, args.packets, 2
    su = L.Setup(ctx, C, 8, 11, [L.FloorTypeOne(1, [0, 128])], [L.Mapping(C)], [L.ModeInfo(False), L.ModeInfo(True)])
    stream = torch.cuda.ExternalStream(ctx.cuda_stream, device=torch.device("cuda", local))

    # synthetic spectrum, device resident before timing: N(0,1)*1e-2, seed 1234 (+rank)
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    spec = torch.randn((S, P, C, N2), generator=gen, device="cuda", dtype=torch.float32) * 1e-2
    stride = P * N2
    pcm = torch.empty((S, C, stride), device="cuda", dtype=torch.float32)
    torch.cuda.synchronize()
    pwrs = [L.PreviousWindowRight(su) for _ in range(S)]
    modes = np.ones(P, np.uint8)
    chains = [L.ChainSpec(pwrs[s], modes, coeff_offset=s * P * C * N2, out_offset=s * C * stride, out_stride=stride)
              for s in range(S)]

    batch = L.Batch(ctx, chains, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, spec.data_ptr(), pcm.data_ptr(),
                    cabi.OUT_F32_PLANAR)
    step = batch.run

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    h0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    host_us = (time.perf_counter() - h0) * 1e6 / args.steps      # host cost of one submission (enqueue only)
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - l0
    dumped = timed_outputs(pcm, batch) if args.dump_outputs and rank == 0 else {}
    # The timed region lasts a few milliseconds (a burst, far below nvidia-smi's sampling period).  The same step is
    # then repeated back to back for >= --sustained-sec, timed the same way: that is the sustained value (power
    # capped clocks), and the window the clock / throttle samples are taken in.
    n_sus = max(args.steps, int(args.sustained_sec * 1e3 / max(ms_total / args.steps, 1e-3)) + 1)
    barrier()
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record(stream)
    for i in range(n_sus):
        step()
        if (i & 255) == 255:
            ctx.synchronize()      # bound the queue depth
    es1.record(stream)
    barrier()
    sus_ms = es0.elapsed_time(es1)
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["sampled"] = f"during the timed steps and the {n_sus} back-to-back steps of the sustained measurement"
    t = torch.tensor([ms_total, sus_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, sus_ms = float(t[0].item()), float(t[1].item())
    ms_step = ms_total / args.steps
    # after warm-up every stream has history: every packet emits 1024 samples per channel
    samples_step = S * P * C * N2 * world
    value = samples_step / (ms_step * 1e-3)

    sustained = {"value": samples_step / (sus_ms / n_sus * 1e-3) / 1e6, "unit": "Msamples/s", "steps": n_sus,
                 "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus}

    # ---- batch scatter + compute + PCM gather (north_star: "NCCL over NVLink used only for the batch scatter/gather") ----
    # The whole batch (world x S streams) starts and ends in rank 0's HBM: grouped ncclSend/ncclRecv out, the same step,
    # grouped ncclSend/ncclRecv back.  Reported beside the compute-only value; the root's link, not the kernels, bounds it.
    with_gather = None
    if world > 1:
        from lewton_b200.sharding import gather_streams, scatter_streams
        n_all = S * world
        spec_all = (torch.randn((n_all, P, C, N2), generator=gen, device="cuda", dtype=torch.float32) * 1e-2) if rank == 0 else None
        pcm_all = torch.empty((n_all, C, stride), device="cuda", dtype=torch.float32) if rank == 0 else None
        g_steps = max(3, min(args.steps, 10))
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(g_steps)]
        with torch.cuda.stream(stream):              # NCCL work is ordered against the library's stream
            for _ in range(2):
                scatter_streams(spec_all, spec, n_all)
                step()
                gather_streams(pcm, pcm_all, n_all)
            barrier()
            for i in range(g_steps):
                ev[i][0].record(stream)
                scatter_streams(spec_all, spec, n_all)
                ev[i][1].record(stream)
                step()
                ev[i][2].record(stream)
                gather_streams(pcm, pcm_all, n_all)
                ev[i][3].record(stream)
            barrier()
        tot = ev[0][0].elapsed_time(ev[-1][3])
        ph = [sum(ev[i][k].elapsed_time(ev[i][k + 1]) for i in range(g_steps)) / g_steps for k in range(3)]
        tg = torch.tensor([tot] + ph, device="cuda", dtype=torch.float64)
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        g_ms = float(tg[0].item()) / g_steps
        moved = (world - 1) * S * P * C * N2 * 4          # bytes the root sends (scatter) and receives (gather) per step
        with_gather = {"value": samples_step / (g_ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": g_ms, "steps": g_steps,
                       "scatter_ms": float(tg[1].item()), "compute_ms": float(tg[2].item()), "gather_ms": float(tg[3].item()),
                       "root_bytes_out_per_step": moved, "root_bytes_in_per_step": moved,
                       "root_scatter_gbs": moved / (float(tg[1].item()) * 1e-3) / 1e9,
                       "root_gather_gbs": moved / (float(tg[3].item()) * 1e-3) / 1e9,
                       "how": "torch.distributed batch_isend_irecv (grouped ncclSend/ncclRecv) on the library's stream; "
                              "the batch starts and ends in rank 0's HBM; phases are max over ranks"}
        del spec_all, pcm_all
    batch.close()
    for p_ in pwrs:
        p_.close()
    del spec, pcm

    # ---- BASELINE.json configs[3] as written: 4096 streams in TOTAL sharded over the ranks (strong scaling) ------
    strong = None
    if args.strong_streams:
        slo, shi = stream_range(args.strong_streams, world, rank)
        Ss, Ps = shi - slo, args.strong_packets
        s_stride = Ps * N2
        s_spec = torch.randn((Ss, Ps, C, N2), generator=gen, device="cuda", dtype=torch.float32) * 1e-2
        s_pcm = torch.empty((Ss, C, s_stride), device="cuda", dtype=torch.float32)
        s_pwrs = [L.PreviousWindowRight(su) for _ in range(Ss)]
        s_modes = np.ones(Ps, np.uint8)
        s_chains = [L.ChainSpec(s_pwrs[s], s_modes, coeff_offset=s * Ps * C * N2, out_offset=s * C * s_stride,
                                out_stride=s_stride) for s in range(Ss)]
        s_batch = L.Batch(ctx, s_chains, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, s_spec.data_ptr(), s_pcm.data_ptr(),
                          cabi.OUT_F32_PLANAR)
        for _ in range(max(args.warmup, 3)):
            s_batch.run()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(args.steps):
            s_batch.run()
        s1.record(stream)
        barrier()
        ts = torch.tensor([s0.elapsed_time(s1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        s_ms = float(ts.item()) / args.steps
        strong = {"value": args.strong_streams * Ps * C * N2 / (s_ms * 1e-3) / 1e6, "unit": "Msamples/s",
                  "scaling": "strong", "streams_total": args.strong_streams, "streams_this_rank": Ss,
                  "packets_per_stream": Ps, "ms_per_step": s_ms,
                  "bytes_in_plus_out_per_gpu": Ss * Ps * C * N2 * 8,
                  "workload": "BASELINE.json configs[3]: batch of 4096 independent stereo streams sharded across the ranks"}
        s_batch.close()
        for p_ in s_pwrs:
            p_.close()
        del s_spec, s_pcm

    # ---- mixed 256/2048 streams (the shape of every 44.1 / 48 kHz Vorbis file): 10 % short blocks in bursts between the
    # long runs, spectrum entry, device-resident; the one-pass schedule of path_mixed.cuh (k_long_s + k_short / k_short_g)
    mixed = None
    if args.mixed_streams:
        Sm, Pm, p_short = args.mixed_streams, 64, 0.10
        rng_m = np.random.default_rng(7 + rank)
        m_seqs, m_offs, c_off = [], [], 0
        for s_ in range(Sm):
            bf = (rng_m.random(Pm) >= p_short).astype(np.uint8)
            bf[0] = bf[-1] = 1                        # the same packets every step on top of the last step's state
            prev, nxt = np.ones(Pm, np.uint8), np.ones(Pm, np.uint8)
            for i in range(Pm):
                if bf[i]:
                    prev[i] = bf[i - 1] if i else 1
                    nxt[i] = bf[i + 1] if i + 1 < Pm else 1
            m_seqs.append((bf, prev, nxt))
            m_offs.append(c_off)
            c_off += int(sum(C * (N2 if b else 128) for b in bf))
        m_spec = torch.randn(c_off, generator=gen, device="cuda", dtype=torch.float32) * 1e-2
        m_pcm = torch.empty(Sm * C * Pm * N2, device="cuda", dtype=torch.float32)
        m_pwrs = [L.PreviousWindowRight(su) for _ in range(Sm)]
        m_chains = [L.ChainSpec(m_pwrs[s_], m_seqs[s_][0], m_seqs[s_][1], m_seqs[s_][2], coeff_offset=m_offs[s_],
                                out_offset=s_ * C * Pm * N2, out_stride=Pm * N2) for s_ in range(Sm)]
        m_batch = L.Batch(ctx, m_chains, cabi.ENTRY_SPECTRUM, cabi.MEM_DEVICE, m_spec.data_ptr(), m_pcm.data_ptr(),
                          cabi.OUT_F32_PLANAR)
        for _ in range(max(args.warmup, 3)):
            m_batch.run()
        barrier()
        launches_m0 = ctx.launch_count
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record(stream)
        for _ in range(args.steps):
            m_batch.run()
        m1.record(stream)
        barrier()
        tm = torch.tensor([m0.elapsed_time(m1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        m_ms = float(tm.item()) / args.steps
        m_samples = c_off            # steady state: every packet emits n/2 samples per channel, i.e. one per coefficient
        mixed = {"value": m_samples * world / (m_ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": m_ms,
                 "streams_per_gpu": Sm, "packets_per_stream": Pm, "short_block_share": p_short,
                 "launches_per_step": (ctx.launch_count - launches_m0) / args.steps,
                 "achieved_gbs": m_samples * 8 / (m_ms * 1e-3) / 1e9,
                 "workload": "stereo 256/2048 streams, bursts of short blocks between long runs, spectrum entry, f32 planar, "
                             "device-resident, state carried from step to step"}
        m_batch.close()
        for p_ in m_pwrs:
            p_.close()
        del m_spec, m_pcm

    # ---- e2e: host (pinned) buffers through the same call --------------------------------------
    Se = min(args.e2e_streams, S)
    h_spec = np.ctypeslib.as_array((np.ctypeslib.ctypes.c_float * (Se * P * C * N2)).from_address(
        cabi.lib().lwb_host_alloc(Se * P * C * N2 * 4)))
    h_pcm = np.ctypeslib.as_array((np.ctypeslib.ctypes.c_float * (Se * C * stride)).from_address(
        cabi.lib().lwb_host_alloc(Se * C * stride * 4)))
    h_spec[:] = (np.random.default_rng(99 + rank).standard_normal(h_spec.size) * 1e-2).astype(np.float32)
    e_pwrs = [L.PreviousWindowRight(su) for _ in range(Se)]
    e_chains = [L.ChainSpec(e_pwrs[s], modes, coeff_offset=s * P * C * N2, out_offset=s * C * stride,
                            out_stride=stride) for s in range(Se)]

    e_batch = L.Batch(ctx, e_chains, cabi.ENTRY_SPECTRUM, cabi.MEM_HOST, h_spec, h_pcm, cabi.OUT_F32_PLANAR)
    e2e_step = e_batch.run

    for _ in range(3):
        e2e_step()
    barrier()
    e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e_steps):
        e2e_step()
    barrier()
    e_sec = time.perf_counter() - t0
    te = torch.tensor([e_sec], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e_sec = float(te.item())
    e2e_value = Se * P * C * N2 * world * e_steps / e_sec

    if rank == 0:
        peak, peak_src = peaks()
        if mixed:
            mixed["frac_of_hbm_peak"] = mixed["achieved_gbs"] / peak
        per_gpu = value / world
        achieved = per_gpu * ALG_BYTES_PER_SAMPLE / 1e9
        traffic, traffic_src = ncu_traffic(S, P)
        line = {"metric": "Msamples/s IMDCT+window+OLA, 2048-pt long blocks", "value": value / 1e6,
                "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "stereo 44.1 kHz long-block (n=2048) packets, batched IMDCT+OLA "
                                       "(BASELINE.json configs[1]); per GPU: streams x packets x 2 channels",
                           "streams_per_gpu": S, "packets_per_stream": P, "channels": C,
                           "bytes_in_per_step_per_gpu": S * P * C * N2 * 4,
                           "l2_policy": "inputs+outputs per step (1 GiB at defaults) exceed the 126 MB L2",
                           "parallelism": f"streams sharded over {world} rank(s), no data-path collective"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write)",
                             "traffic_source": traffic_src, "algorithmic_bytes_per_launch": S * P * C * N2 * ALG_BYTES_PER_SAMPLE,
                             "peak_source": peak_src,
                             "kernel": "k_long", "algorithmic_bytes_per_sample": ALG_BYTES_PER_SAMPLE},
                "e2e": {"value": e2e_value / 1e6, "unit": "Msamples/s",
                        "h2d_bytes_per_step": Se * P * C * N2 * 4, "d2h_bytes_per_step": Se * C * stride * 4,
                        "streams": Se, "steps": e_steps, "timer": "host wall clock around synchronous calls"},
                "sustained": sustained, "strong_scaling": strong, "with_gather": with_gather, "mixed_streams": mixed,
                "gpu_launches": int(launches), "host_enqueue_us_per_step": host_us, "clocks": clocks,
                "host_binding": {"numa_node": int(numa), "cpus": len(os.sched_getaffinity(0)),
                                 "how": "lwb_bind_host_to_device: CPU affinity + preferred memory node of the GPU's PCIe root"}}
        if not args.no_cpu_baseline:
            os.sched_setaffinity(0, affinity0)        # the CPU arm gets every core the container has
            cabi.lib().lwb_bind_host_to_device(-1)    # ... and the default memory policy
            threads = host_threads()
            v1, _, _ = cpu_reference(8, 17, 1, target_sec=0.5)
            v, sec, reps = cpu_reference(8 * threads, 17, threads, target_sec=2.0)
            line["cpu_baseline"] = {"value": v / 1e6, "unit": "Msamples/s", "cores": threads, "kind": "port",
                                    "single_thread_value": v1 / 1e6,
                                    "sample": f"{8 * threads} stereo streams x 17 long packets swept {reps}x = "
                                              f"{sec:.2f} s wall on {threads} threads ({sec * threads:.0f} core-s); "
                                              "lewton-equivalent C restatement (oracle/), the crate itself is Rust"}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dumped:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
