#!/usr/bin/env python
"""pcm_ingest.py — what PCM ingest buys the EBUr128 cycle: host-path end-to-end rate per input format, device-path cycle
with and without the conversion, and the conversion kernel alone.

    python profiles/pcm_ingest.py [--steps 300] [--rounds 5] [--out FILE] [--trace DIR]

Workload: bench.py's e2e leg — 8192 stereo instances, 48 kHz, 1024-frame cycles, integration running, dBTP in tolerance mode
(B200M_PREC_FMA); one step = run + b200m_r128_results (D2H of the readings inside the timed region).

* host path: F32 planar (b200m_r128_run_host, today's path), S16 / S24 / S32 interleaved (b200m_r128_run_host_pcm), each from
  two alternating pinned blocks of b200m_host_alloc; the arms are timed in turn, `--rounds` times, `--steps` steps each.
* device path: b200m_r128_run_device_pcm on an S16 interleaved ring against b200m_r128_run_device on the float32 ring of the
  same values (8 distinct blocks each, larger than L2), CUDA events, arms alternated.
* the conversion alone (b200m_pcm_convert, interleaved S16 / S24 / S32 -> planar float32 rows), CUDA events; its bytes
  (read + write) over time, against the data sheet's HBM bandwidth and a device-to-device copy measured in the same run.

Every arm is fed the same 16-bit values (S24 = v << 8, S32 = v << 16, F32 = v * 2^-15: one float32 each way), so all banks
of a leg end bit-identical; the script checks that.  --trace DIR records a few steps of each host arm with torch.profiler.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_INST, NFRAM, RING = 8192, 1024, 8
SAMPLES = 2 * N_INST * NFRAM
HBM_DATASHEET_GBS = 7700.0          # HGX B200 data sheet, one GPU


def gpu_meta():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as e:                                       # the numbers stand without it, but say so
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def values(rng, n_blocks):
    """int16 [n_inst, n_blocks * NFRAM, 2]: noise at per-channel levels -6 .. -36 dBFS (bench.py's ring)"""
    c = np.arange(2 * N_INST).reshape(N_INST, 1, 2)
    gain = 10.0 ** (-(6.0 + 30.0 * (c % 97) / 96.0) / 20.0)
    x = rng.uniform(-1.0, 1.0, (N_INST, n_blocks * NFRAM, 2)) * gain
    return np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)


def formats(v):
    """the same values as each arm's array: {name: (fmt, array)}; F32 planar [2N, nfram], the others interleaved"""
    import meters_lv2_b200 as B
    w = v.astype(np.int32)
    s24 = np.ascontiguousarray((w << 8).astype("<i4").view(np.uint8).reshape(*v.shape, 4)[..., :3])
    return {"f32_planar": (B.PCM_F32 | B.PCM_PLANAR, np.ascontiguousarray((v.astype(np.float32) * np.float32(2.0 ** -15)).transpose(0, 2, 1)).reshape(2 * N_INST, -1)),
            "s16_interleaved": (B.PCM_S16 | B.PCM_INTERLEAVED, v),
            "s24_interleaved": (B.PCM_S24 | B.PCM_INTERLEAVED, s24),
            "s32_interleaved": (B.PCM_S32 | B.PCM_INTERLEAVED, w << 16)}


def pinned_like(a):
    import meters_lv2_b200 as B
    p = B.host_alloc(1, a.nbytes // 4).view(a.dtype).reshape(a.shape)
    p[:] = a
    return p


def new_bank():
    import meters_lv2_b200 as B
    g = B.EBUr128(N_INST, 48000.0, dbtp_enable=True)
    g.set_precision(B.PREC_FMA)
    g.control(B.EBUr128.START)
    return g


def same_state(banks):
    """checkpoint blobs equal; written into zeroed buffers, since the blob's alignment padding is left unwritten"""
    import meters_lv2_b200 as B

    def blob(g):
        n = B.lib().b200m_r128_snapshot_size(g.h)
        buf = np.zeros(n, np.uint8)
        B._ck(B.lib().b200m_r128_snapshot(g.h, B._np_ptr(buf), n, B._stream_ptr(None)))
        return buf
    ref = blob(banks[0])
    return all(np.array_equal(ref, blob(b)) for b in banks[1:])


def host_leg(args, out):
    import torch
    import meters_lv2_b200 as B
    rng = np.random.default_rng(0x42B200)
    v = values(rng, 2)
    arms = {}
    for name, (fmt, a) in formats(v).items():
        blocks = [pinned_like(a[:, b * NFRAM:(b + 1) * NFRAM]) for b in range(2)]
        arms[name] = dict(fmt=fmt, blocks=blocks, ptrs=[b.ctypes.data for b in blocks], bank=new_bank(), secs=[], bytes=blocks[0].nbytes)
    res = np.empty(N_INST, B.EBU_RESULT_DTYPE); tp = np.empty(N_INST, np.float32)

    def step(arm, s):
        arm["bank"].run_pcm_ptr(arm["ptrs"][s % 2], arm["fmt"], NFRAM, NFRAM, host=True)
        arm["bank"].results(out=res, tp=tp)

    for arm in arms.values():
        for s in range(5):
            step(arm, s)
    for r in range(args.rounds):
        for arm in arms.values():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for s in range(args.steps):
                step(arm, s)
            torch.cuda.synchronize()
            arm["secs"].append(time.perf_counter() - t0)
    f32 = None
    leg = {}
    for name, arm in arms.items():
        per = [args.steps * SAMPLES / t for t in arm["secs"]]
        rate = args.steps * args.rounds * SAMPLES / sum(arm["secs"])
        f32 = f32 or rate
        leg[name] = {"samples_per_s": rate, "per_round": per, "ms_per_step": sum(arm["secs"]) / (args.steps * args.rounds) * 1e3,
                     "h2d_bytes_per_step": arm["bytes"], "h2d_gbs": arm["bytes"] * args.steps * args.rounds / sum(arm["secs"]) / 1e9,
                     "vs_f32_planar": rate / f32, "timed_seconds": sum(arm["secs"])}
    leg["banks_bit_identical"] = same_state([a["bank"] for a in arms.values()])
    out["host_path"] = leg
    if args.trace:
        trace_host(args, arms, step)
    for a in arms.values():
        a["bank"].close()


def trace_host(args, arms, step):
    import torch
    from torch.profiler import ProfilerActivity, profile
    os.makedirs(args.trace, exist_ok=True)
    for name, arm in arms.items():
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for s in range(6):
                step(arm, s)
            torch.cuda.synchronize()
        prof.export_chrome_trace(os.path.join(args.trace, "pcm_%s.pt.trace.json" % name))
        with open(os.path.join(args.trace, "pcm_%s.txt" % name), "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25))


def timed(fn, steps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for s in range(steps):
        fn(s)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def device_leg(args, out):
    import torch
    import meters_lv2_b200 as B
    rng = np.random.default_rng(0x42B201)
    v = values(rng, RING)                                              # [N, RING * NFRAM, 2] int16
    fm = formats(v)
    d = {k: torch.from_numpy(np.ascontiguousarray(a)).cuda() for k, (_, a) in fm.items()}
    del fm
    ring_frames = RING * NFRAM
    bps = {"s16_interleaved": 2, "s24_interleaved": 3, "s32_interleaved": 4}

    def blk(name, s):
        t = d[name]
        step = 4 if name == "f32_planar" else 2 * bps[name]
        return t.data_ptr() + step * NFRAM * (s % RING)

    # the cycle: run_device on the float ring vs run_device_pcm on the S16 ring of the same values
    banks = {"f32_planar": new_bank(), "s16_interleaved": new_bank()}
    fmt = {"f32_planar": B.PCM_F32 | B.PCM_PLANAR, "s16_interleaved": B.PCM_S16 | B.PCM_INTERLEAVED}
    ms = {k: [] for k in banks}
    for k in banks:
        timed(lambda s: banks[k].run_pcm_ptr(blk(k, s), fmt[k], ring_frames, NFRAM), 2 * RING)
    for r in range(args.rounds):
        for k in banks:
            ms[k].append(timed(lambda s: banks[k].run_pcm_ptr(blk(k, s), fmt[k], ring_frames, NFRAM), args.steps))
    cyc = {k: {"ms_per_step": float(np.median(m)), "per_round_ms": m, "samples_per_s": SAMPLES / (np.median(m) * 1e-3)} for k, m in ms.items()}
    cyc["conversion_share_of_cycle"] = 1.0 - cyc["f32_planar"]["ms_per_step"] / cyc["s16_interleaved"]["ms_per_step"]
    cyc["banks_bit_identical"] = same_state(list(banks.values()))
    out["device_path"] = cyc
    for g in banks.values():
        g.close()

    # the conversion kernel alone, and a device-to-device copy of 512 MiB as the practical HBM ceiling of this run
    dst = torch.empty((2 * N_INST, NFRAM), dtype=torch.float32, device="cuda")
    conv = {}
    for name in ("s16_interleaved", "s24_interleaved", "s32_interleaved"):
        f = {"s16_interleaved": B.PCM_S16, "s24_interleaved": B.PCM_S24, "s32_interleaved": B.PCM_S32}[name] | B.PCM_INTERLEAVED

        def go(s, name=name, f=f):
            import ctypes as C
            rc = B.lib().b200m_pcm_convert(0, C.c_void_p(blk(name, s)), f, 2, N_INST, ring_frames, NFRAM, C.c_void_p(dst.data_ptr()), NFRAM, None)
            assert rc == 0, B.lib().b200m_last_error()
        timed(go, 2 * RING)
        m = float(np.median([timed(go, args.steps) for _ in range(args.rounds)]))
        nbytes = SAMPLES * (bps[name] + 4)
        conv[name] = {"ms": m, "bytes_read_plus_written": nbytes, "gbs": nbytes / (m * 1e-3) / 1e9,
                      "share_of_datasheet_hbm": nbytes / (m * 1e-3) / 1e9 / HBM_DATASHEET_GBS}
    a = torch.empty(128 << 20, dtype=torch.float32, device="cuda"); b = torch.empty_like(a)
    timed(lambda s: b.copy_(a), 3)
    mc = float(np.median([timed(lambda s: b.copy_(a), 20) for _ in range(args.rounds)]))
    copy_gbs = 2 * a.numel() * 4 / (mc * 1e-3) / 1e9
    for c in conv.values():
        c["share_of_measured_copy"] = c["gbs"] / copy_gbs
    out["conversion_kernel"] = conv
    out["d2d_copy_gbs"] = copy_gbs
    out["hbm_datasheet_gbs"] = HBM_DATASHEET_GBS


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--trace", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pcm_ingest.py: no CUDA device")
    out = {"config": {"instances": N_INST, "channels_per_instance": 2, "block": NFRAM, "fs": 48000.0, "precision": "B200M_PREC_FMA",
                      "steps": args.steps, "rounds": args.rounds, "step": "run + b200m_r128_results"}}
    out["meta"] = gpu_meta()
    host_leg(args, out)
    device_leg(args, out)
    h = out["host_path"]
    out["acceptance"] = {"s16_vs_f32": h["s16_interleaved"]["vs_f32_planar"], "s24_vs_f32": h["s24_interleaved"]["vs_f32_planar"],
                         "s32_vs_f32": h["s32_interleaved"]["vs_f32_planar"]}
    s = json.dumps(out, indent=1)
    print(s, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
