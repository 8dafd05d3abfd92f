#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native metering engine (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Workload (BASELINE.json `metric`: "audio-samples/sec/GPU (48 kHz stereo, 8192-ch batch) EBU R128 + true-peak"):
8192 stereo instances PER GPU (weak scaling), 48 kHz, 1024-frame blocks, the EBUr128 plugin's audio cycle with
integration running and dBTP enabled (src/ebulv2.cc:341-367: Ebu_r128_proc::process + TruePeakdsp::process_max on
both channels + getters).  One "step" = one such cycle over the whole batch = 16 777 216 mono samples per GPU.

`value`  = samples/s summed over all N GPUs, input resident in HBM (ring of 8 distinct 64 MiB blocks > L2), the dBTP FIR in
           the engine's tolerance mode (B200M_PREC_FMA: readings within +-1e-4 dB of the reference, the contract's float
           tolerance; EBU R128 floats and histograms bit-exact).  `value_bit_exact` = the same cycle with every float
           bit-identical to the reference (B200M_PREC_EXACT, the library default).
`e2e`    = the same cycle through b200m_r128_run_host with pinned HOST buffers, H2D copy and D2H result read inside the
           timed region (PCIe-bound: 64 MiB per cycle cannot shrink, the LV2 contract is float32 audio).
`--impl reference` times the reference's own CPU code (oracle/_ref, else the oracle port) on every CPU the process may use.
`--dump-outputs DIR` writes what the headline's last timed step left for its caller (b200m_r128_results on rank 0: the nine
EBU R128 readings, histogram counts and fragment power of every instance, and the dBTP hold) as DIR/<field>.npy; the input
ring is seeded, so two builds run with the same arguments can be compared output for output.

The JSON line is printed (and flushed) as soon as the headline, e2e, roofline and cpu_baseline exist; the other BASELINE
configs, the whole-mix all-reduce and the parity spot check run afterwards and the enriched line is printed again
(the last line supersedes the first; both are complete on their own).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "audio-samples/sec/GPU (48 kHz stereo, 8192-ch batch) EBU R128 + true-peak"
FS = 48000.0
N_INST = 8192          # stereo instances per GPU
NFRAM = 1024
RING = 8               # distinct device-resident blocks: 8 x 64 MiB = 512 MiB > 126 MB L2
PRIME = 480            # untimed blocks (10.2 s of audio) so that S, I (>=50 M-points) and LRA (>=20 S-points) are live
SAMPLES_PER_STEP = N_INST * 2 * NFRAM
CPU_BLOCKS = 4         # blocks per CPU step


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bf16_peak_tflops():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p)).get("bf16_tflops", 0.0)) or None
    return None


def traffic_for(kernel):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(kernel)
    return None


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons of one GPU through NVML while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.maxc = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.maxc = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        names = {"GpuIdle": 0x1, "ApplicationsClocksSetting": 0x2, "sw_power_cap": 0x4, "hw_slowdown": 0x8,
                 "SyncBoost": 0x10, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80}
        while not self.stop_flag:
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, v in names.items():
                    if r & v and k != "GpuIdle":
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.maxc, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.maxc, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def dist_env():
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), ws


def make_ring(torch, dev, rank):
    g = torch.Generator(device=dev); g.manual_seed(0x42B200 + rank)
    c = torch.arange(2 * N_INST, device=dev)
    gain = torch.pow(10.0, -(6.0 + 30.0 * (c % 97).float() / 96.0) / 20.0)
    x = (torch.rand((2 * N_INST, RING * NFRAM), generator=g, device=dev, dtype=torch.float32) * 2 - 1) * gain[:, None]
    return x.contiguous()


def timed_loop(torch, dist, ws, fn, steps):
    """barrier + synchronize on both sides, CUDA events on the current stream, max over ranks (ms)"""
    if ws > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        fn(s)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if ws > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    return ms


def emit(out):
    print(json.dumps(out), flush=True)


def run_b200(args):
    import torch
    import torch.distributed as dist
    import meters_lv2_b200 as B
    rank, local, ws = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if ws > 1:
        dist.init_process_group("nccl", device_id=dev)      # NCCL_DEBUG is left exactly as the caller set it
    K, W = args.steps, max(args.warmup, 3)
    hbm_peak, peak_src = peaks()
    bf16_peak = bf16_peak_tflops()
    x = make_ring(torch, dev, rank)
    stride = x.stride(0)
    base = x.data_ptr()

    def blk(s):
        return base + 4 * NFRAM * (s % RING)

    # ---- headline: the EBUr128 audio cycle, device-resident input -------------------------------------------------
    bank = B.EBUr128(N_INST, FS, dbtp_enable=True, device=local)
    bank.control(B.EBUr128.START)
    bank.set_precision(B.PREC_FMA)
    pos = [0]

    def step(_):
        bank.run_ptr(blk(pos[0]), stride, NFRAM)
        pos[0] += 1

    # clocks / throttle reasons are sampled from the priming blocks on (same kernels, same load): the timed region of a 20-step run
    # lasts 2 ms, too short for NVML on its own
    sampler = ClockSampler(local); sampler.start()
    for s in range(PRIME + W):
        step(s)
    torch.cuda.synchronize()
    l0 = B.launch_count()
    ms = timed_loop(torch, dist, ws, step, K)
    launches = B.launch_count() - l0
    sampler.stop_flag = True; sampler.join()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *bank.results())
    value = ws * SAMPLES_PER_STEP * K / (ms * 1e-3)
    bank.set_precision(B.PREC_EXACT)
    for s in range(W):
        step(s)
    ms_exact = timed_loop(torch, dist, ws, step, K)
    blocks_run = pos[0]

    out = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": ws, "steps": K, "warmup": W,
           "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "impl": "b200",
           "config": {"workload": "8192 stereo EBU R128 M+S+I (integrating) + dBTP true-peak 4x (ebur128_run audio cycle) per GPU",
                      "instances_per_gpu": N_INST, "channels_per_instance": 2, "block": NFRAM, "fs": FS,
                      "value_is": "aggregate over all %d GPUs (samples/s); value_per_gpu = value / n_gpus" % ws,
                      "precision": "dBTP FIR in tolerance mode B200M_PREC_FMA: on the tensor cores as a 3xTF32 Toeplitz GEMM (fp32 accumulate; "
                                   "readings within 1e-5 dB of the reference measured, +-1e-4 dB is the contract's float tolerance; "
                                   "tests/test_tpk_fma_gpu.py); EBU R128 floats + histograms bit-exact (fp32, unfused); "
                                   "value_bit_exact = all floats bit-identical (B200M_PREC_EXACT, library default)",
                      "input": "device ring of %d distinct 64 MiB blocks (512 MiB > L2), no L2 flush needed" % RING,
                      "prime_blocks": PRIME, "parallelism": "channel-shard x%d, no data-path collective" % ws},
           "value_per_gpu": value / ws, "value_bit_exact": ws * SAMPLES_PER_STEP * K / (ms_exact * 1e-3), "ms_per_step_bit_exact": ms_exact / K,
           "gpu_launches": int(launches), "clocks": sampler.summary()}

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region ---------------------------------
    hbank = B.EBUr128(N_INST, FS, dbtp_enable=True, device=local)
    hbank.control(B.EBUr128.START)
    hbank.set_precision(B.PREC_FMA)
    HR = 2
    # HR separate dense [channels][1024] blocks from the library's pinned allocator (GPU-local NUMA node): what a host
    # that double-buffers its capture hands over each cycle; dense blocks go over PCIe as one DMA per slice
    hosts = [B.host_alloc(2 * N_INST, NFRAM) for _ in range(HR)]
    for i, hb in enumerate(hosts):
        hb[:] = x[:, i * NFRAM:(i + 1) * NFRAM].cpu().numpy()
    res_buf = np.empty(N_INST, B.EBU_RESULT_DTYPE); tp_buf = np.empty(N_INST, np.float32)
    hptrs = [hb.ctypes.data for hb in hosts]
    ke = max(3, min(K, args.e2e_steps))

    def estep(s):
        hbank.run_ptr(hptrs[s % HR], NFRAM, NFRAM, host=True)
        hbank.results(out=res_buf, tp=tp_buf)

    for s in range(3):
        estep(s)
    if ws > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(ke):
        estep(s)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if ws > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    h2d = 2 * N_INST * NFRAM * 4
    out["e2e"] = {"value": ws * SAMPLES_PER_STEP * ke / dt, "unit": "samples/s", "steps": ke, "ms_per_step": dt / ke * 1e3,
                  "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(res_buf.nbytes + tp_buf.nbytes),
                  "pcie_gbs_per_gpu": h2d * ke / dt / 1e9,
                  "api": "b200m_r128_run_host + b200m_r128_results (pinned host buffers from b200m_host_alloc)",
                  "bound": "PCIe host->device: 64 MiB of float32 audio per cycle and GPU (the LV2 port format), copy and kernels overlapped in 4 slices; "
                           "the kernels need %.0f%% of the step" % (100.0 * (ms / K) / (dt / ke * 1e3))}
    del hbank

    # ---- per-kernel timings for the roofline (kernel alone, same ring, CUDA events) -----------------------------
    # the same FIR on the CUDA cores (tpmax_kernel<IMM,FMA>), for the record: the tensor-core kernel is the default for banks this size
    os.environ["B200M_TPK_TC"] = "0"
    tpc = B.TruePeakKmeter(2 * N_INST, FS, flags=B.TPK_TRUEPEAK, device=local)
    tpc.set_precision(B.PREC_FMA)
    for s in range(W):
        tpc.process_ptr(blk(s), stride, NFRAM, B.TP_MODE_MAX)
    ms_tpc = timed_loop(torch, dist, ws, lambda s: tpc.process_ptr(blk(s), stride, NFRAM, B.TP_MODE_MAX), K)
    del tpc
    os.environ.pop("B200M_TPK_TC", None)
    tpb = B.TruePeakKmeter(2 * N_INST, FS, flags=B.TPK_TRUEPEAK, device=local)
    tpb.set_precision(B.PREC_FMA)
    ebb = B.Ebu_r128_proc(N_INST, 2, FS, device=local); ebb.integr_start()
    for s in range(W):
        tpb.process_ptr(blk(s), stride, NFRAM, B.TP_MODE_MAX)
        ebb.process_ptr(blk(s), stride, NFRAM)
    ms_tp = timed_loop(torch, dist, ws, lambda s: tpb.process_ptr(blk(s), stride, NFRAM, B.TP_MODE_MAX), K)
    tpb.set_precision(B.PREC_EXACT)
    for s in range(W):
        tpb.process_ptr(blk(s), stride, NFRAM, B.TP_MODE_MAX)
    ms_tpx = timed_loop(torch, dist, ws, lambda s: tpb.process_ptr(blk(s), stride, NFRAM, B.TP_MODE_MAX), K)
    l1 = B.launch_count()
    ms_eb = timed_loop(torch, dist, ws, lambda s: ebb.process_ptr(blk(s), stride, NFRAM), K)
    eb_launch = B.launch_count() - l1
    fp32_peak = B.peak_probe(0, local)                      # unfused FMUL+FADD lane-ops/s = FFMA issue rate (one fma-pipe instruction per lane and clock)
    alg_bytes = SAMPLES_PER_STEP * 4.0                      # 4 B per mono sample read once (SURVEY §8d); outputs ~0
    tp_gbs = alg_bytes / (ms_tp / K * 1e-3) / 1e9
    tpx_gbs = alg_bytes / (ms_tpx / K * 1e-3) / 1e9
    eb_gbs = alg_bytes / (ms_eb / K * 1e-3) / 1e9
    # fp32 instructions the FIR executes per input sample: tolerance mode 120 (72 FFMA + 48 FADD, csrc/tpk.cu fir16_fma);
    # exact mode 288 unfused FMUL/FADD for phases 1-3 (+96 for phase 0 where the exact-delay guard fails: never on this noise)
    out["roofline"] = {"kernel": "tpmax_tc_kernel (4x polyphase FIR as a Toeplitz GEMM on tcgen05 kind::tf32 with the 3xTF32 split, + max; tolerance mode)",
                       "bound": "hbm", "achieved": tp_gbs, "peak": hbm_peak,
                       "unit": "GB/s", "frac": tp_gbs / hbm_peak, "traffic": traffic_for("tpmax_tc_kernel"), "peak_source": peak_src,
                       "ms_per_launch": ms_tp / K, "algorithmic_bytes_per_launch": alg_bytes,
                       "note": "bound by its producer / epilogue warps (window -> {hi, lo} -> TMEM, TMEM -> maxima), not by HBM or the tensor pipe, see roofline_tensor and DESIGN.md; share of the cycle: %.0f%%" % (100.0 * ms_tp / ms)}
    # executed tensor-core work: per [8 channels x 256 samples] tile 8 K-steps x (128 x 96 x 8 + 128 x 48 x 8) MACs (25 % of the Toeplitz B is zero,
    # and the three products of the split count three times): 1152 flop per input sample, of which 288 (3 phases x 48 taps x 2) are the FIR's own
    tf32_peak = (bf16_peak / 2.0) if bf16_peak else None
    tc_tflops = SAMPLES_PER_STEP * 1152.0 / (ms_tp / K * 1e-3) / 1e12
    out["roofline_tensor"] = {"kernel": "tpmax_tc_kernel", "bound": "tensor (kind::tf32)", "achieved": tc_tflops, "peak": tf32_peak, "unit": "TFLOP/s",
                              "frac": (tc_tflops / tf32_peak) if tf32_peak else None, "executed_flop_per_sample": 1152, "fir_flop_per_sample": 288,
                              "peak_source": "half of MEASURED_PEAKS.json's dense bf16 rate (tf32 runs at half the bf16 rate)" if tf32_peak else "none"}
    out["roofline_alu"] = {"kernel": "tpmax_kernel<IMM,FMA> (the same FIR on the CUDA cores: B200M_TPK_TC=0, and every bank too small for the tensor-core grid)",
                           "bound": "fp32 issue (fma pipe)", "achieved": SAMPLES_PER_STEP * 120.0 / (ms_tpc / K * 1e-3) / 1e9,
                           "peak": fp32_peak, "unit": "1e9 lane-ops/s", "frac": SAMPLES_PER_STEP * 120.0 / (ms_tpc / K * 1e-3) / 1e9 / fp32_peak,
                           "ops_per_sample": 120, "ms_per_launch": ms_tpc / K, "hbm_frac": alg_bytes / (ms_tpc / K * 1e-3) / 1e9 / hbm_peak,
                           "peak_source": "b200m_peak_probe(0) measured in this run",
                           "bit_exact_mode": {"ops_per_sample": 288, "ms_per_launch": ms_tpx / K, "hbm_frac": tpx_gbs / hbm_peak,
                                              "frac": SAMPLES_PER_STEP * 288.0 / (ms_tpx / K * 1e-3) / 1e9 / fp32_peak}}
    out["roofline_kernels"] = [
        {"kernel": "ebu_kweight_frag (+ebu_fragment_kernel every 2400 frames)", "bound": "hbm", "achieved": eb_gbs, "peak": hbm_peak, "unit": "GB/s",
         "frac": eb_gbs / hbm_peak, "traffic": traffic_for("ebu_kweight_frag"), "ms_per_block": ms_eb / K, "launches_per_block": eb_launch / K,
         "samples_per_s": SAMPLES_PER_STEP * K / (ms_eb * 1e-3)}]
    del tpb, ebb

    # ---- CPU baseline beside it (rank 0; the other ranks wait at the next collective) ---------------------------
    if rank == 0 and not args.no_cpu:
        try:
            out["cpu_baseline"] = cpu_baseline(budget_s=8.0)
        except Exception as e:
            out["cpu_baseline"] = {"error": repr(e)}
    if rank == 0:
        emit(out)                                            # complete on its own; everything below only adds keys

    if not args.headline_only:
        # ---- whole-mix gated loudness (the path's one exchange, SURVEY §8e): per-GPU histogram sum -> ONE int32[1508]
        # all-reduce (NCCL when N > 1) -> calc_integ / calc_range on the sum.  Due once per 0.5 s of audio, not per cycle.
        try:
            from meters_lv2_b200 import shard
            mixv = torch.zeros(B.MIX_WORDS, dtype=torch.int32, device=dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(3):                                   # first calls set up the communicator
                bank.ebu.mix_reduce(mixv); shard.allreduce_mix(mixv)
            torch.cuda.synchronize(); e0.record()
            bank.ebu.mix_reduce(mixv); shard.allreduce_mix(mixv)
            e1.record(); torch.cuda.synchronize()
            mo = bank.ebu.mix_finish(mixv)
            cm = int(mixv[2 * 752].item()); res0, _tp0 = bank.results()
            out["whole_mix"] = {"integrated": float(mo[0]), "range_min": float(mo[2]), "range_max": float(mo[3]),
                                "hist_M_points": cm, "hist_M_points_rank0_times_n": int(res0["hist_M_count"].astype(np.int64).sum()) * ws,
                                "reduce_plus_allreduce_us": e0.elapsed_time(e1) * 1e3, "collective": "nccl all_reduce int32[%d]" % B.MIX_WORDS if ws > 1 else "none (N = 1)"}
        except Exception as e:
            out["whole_mix"] = {"error": repr(e)}

        # ---- parity spot check against the CPU oracle on the first instances (same block sequence) ----------------
        if rank == 0:
            try:
                out["parity"] = spot_check(B, bank, x, blocks_run)
            except Exception as e:  # the bench number stands on its own; tests are the parity gate
                out["parity"] = {"error": repr(e)}
        del bank

        # ---- the other BASELINE configs (reported, not the headline) ------------------------------------------------
        try:
            out["configs"] = other_configs(torch, dist, B, x, K, W, hbm_peak, ws, local)
        except Exception as e:
            out["configs"] = {"error": repr(e)}
        if rank == 0:
            emit(out)
    if ws > 1:
        dist.destroy_process_group()


def dump_outputs(d, res, tp):
    """one .npy per result field (float32; the int32 counts as float64, exactly) plus tp_max.npy: 8192 instances, < 1 MB in all"""
    os.makedirs(d, exist_ok=True)
    for name in res.dtype.names:
        v = res[name]
        np.save(os.path.join(d, name + ".npy"), v.astype(np.float64 if v.dtype.kind == "i" else np.float32))
    np.save(os.path.join(d, "tp_max.npy"), tp.astype(np.float32))


def spot_check(B, bank, x, blocks_run, ni=2):
    import _oracle as O
    xs = x[:2 * ni].cpu().numpy()
    oe = O.Ebu(ni, 2, FS); ot = O.TruePeak(2 * ni, FS); oe.integr("start")
    tpmax = np.full(ni, -np.inf, np.float32)
    for s in range(blocks_run):
        b = s % RING
        blkx = np.ascontiguousarray(xs[:, b * NFRAM:(b + 1) * NFRAM])
        oe.process(blkx); ot.process(blkx, mode=1)
        m, _ = ot.read()
        v = np.maximum(m[0::2], m[1::2])
        with np.errstate(divide="ignore"):
            tp = np.where(v == 0, -np.inf, (20.0 * np.log10(v.astype(np.float32)).astype(np.float64)).astype(np.float32))
        tpmax = np.maximum(tpmax, tp)
    res, tpg = bank.results()
    orr = oe.read()
    names = ("loudness_M", "maxloudn_M", "loudness_S", "maxloudn_S", "integrated", "integ_thr", "range_min", "range_max", "range_thr")
    exact = all(np.array_equal(res[n][:ni].view(np.uint32), orr[:, i].view(np.uint32)) for i, n in enumerate(names))
    hm, hs = bank.ebu.histogram(0); om, os_, _ = oe.hist(0)
    return {"oracle": O.load().orc_kind().decode(), "instances_checked": ni, "blocks": blocks_run,
            "ebu_bit_exact": bool(exact), "hist_bit_exact": bool(np.array_equal(hm, om) and np.array_equal(hs, os_)),
            "dbtp_max_abs_diff_db": float(np.max(np.abs(tpg[:ni].astype(np.float64) - tpmax.astype(np.float64)))), "dbtp_tolerance_db": 1e-4}


def other_configs(torch, dist, B, x, K, W, hbm_peak, ws, local):
    """BASELINE.json configs[1..4].  N = 1: each at its stated size on this GPU.  N > 1: C3 and C5 with the TOTAL batch
    BASELINE names split over the ranks (strong scaling: 8192 / N resp. 2048 / N stereo instances per GPU), timed as the
    max over ranks; throughput = total units / that time."""
    base, stride = x.data_ptr(), x.stride(0)
    cfg = {}

    def blk(s):
        return base + 4 * NFRAM * (s % RING)

    if ws == 1:
        # C2 pure: EBU R128 only
        e = B.Ebu_r128_proc(N_INST, 2, FS, device=local); e.integr_start()
        for s in range(PRIME // 4 + W):
            e.process_ptr(blk(s), stride, NFRAM)
        ms = timed_loop(torch, dist, 1, lambda s: e.process_ptr(blk(s), stride, NFRAM), K)
        n = N_INST * 2 * NFRAM
        cfg["C2_ebu_r128_8192st"] = {"samples_per_s": n * K / (ms * 1e-3), "ms_per_block": ms / K, "hbm_frac": n * 4 * K / (ms * 1e-3) / 1e9 / hbm_peak}
        del e

    # C3: true peak (process) + K-meter, read every block (TPnRMS, src/dr14.c:391-450); 8192 stereo in total
    n3 = 2 * (N_INST // ws)
    for prec, tag in ((B.PREC_FMA, "C3_truepeak_k20_8192st"), (B.PREC_EXACT, "C3_truepeak_k20_8192st_bit_exact")):
        t = B.TruePeakKmeter(n3, FS, device=local); t.set_precision(prec)

        def c3(s):
            t.process_ptr(blk(s), stride, NFRAM); t.read_device()
        for s in range(W):
            c3(s)
        ms = timed_loop(torch, dist, ws, c3, K)
        n = ws * n3 * NFRAM
        cfg[tag] = {"samples_per_s": n * K / (ms * 1e-3), "ms_per_block": ms / K, "hbm_frac_per_gpu": n / ws * 4 * K / (ms * 1e-3) / 1e9 / hbm_peak,
                    "stereo_instances_per_gpu": n3 // 2, "scaling": "strong" if ws > 1 else "single GPU"}
        del t

    if ws == 1:
        # C4: 4096 stereo 30-band spectrum (unit: stereo frames)
        fp64_peak = B.peak_probe(1, local)
        sp = B.Spectr30(4096, 2, FS, device=local)
        k4 = max(3, K // 10)
        for s in range(2):
            sp.process_ptr(blk(s), stride, NFRAM)
        ms = timed_loop(torch, dist, 1, lambda s: sp.process_ptr(blk(s), stride, NFRAM), k4)
        fr = 4096 * NFRAM
        c4x = {"frames_per_s": fr * k4 / (ms * 1e-3), "ms_per_block": ms / k4, "hbm_frac": fr * 8 * k4 / (ms * 1e-3) / 1e9 / hbm_peak,
               "fp64_frac": fr * 30 * 39.0 * k4 / (ms * 1e-3) / 1e9 / fp64_peak, "fp64_ops_per_frame_and_band": 39}
        sp.set_precision(B.PREC_FMA)                          # fused multiply-adds: 25 fp64 instructions per frame and band, levels within +-1e-4 dB
        for s in range(2):
            sp.process_ptr(blk(s), stride, NFRAM)
        ms = timed_loop(torch, dist, 1, lambda s: sp.process_ptr(blk(s), stride, NFRAM), k4)
        cfg["C4_spectr30_4096st"] = {"frames_per_s": fr * k4 / (ms * 1e-3), "ms_per_block": ms / k4, "hbm_frac": fr * 8 * k4 / (ms * 1e-3) / 1e9 / hbm_peak,
                                     "fp64_frac": fr * 30 * 25.0 * k4 / (ms * 1e-3) / 1e9 / fp64_peak, "fp64_ops_per_frame_and_band": 25,
                                     "precision": "B200M_PREC_FMA (band levels within +-1e-4 dB)", "fp64_peak_glops": fp64_peak, "bit_exact": c4x}
        del sp

    # C5: 2048 stereo phasewheel 2048-pt FFT + Stcorr in total (unit: stereo frames)
    n5 = 2048 // ws
    cfg["C5_phasewheel_stcorr_2048st"] = c5_config(torch, dist, B, blk, stride, K, W, hbm_peak, ws, local, n5)
    return cfg


def c5_config(torch, dist, B, blk, stride, K, W, hbm_peak, ws, local, n5):
    """fused feed (one kernel reads the block once: Stcorrdsp + FFT ring append) + the 25 Hz analysis kernel.  Headline of this config:
    the correlation in its time-parallel tolerance mode (B200M_PREC_FMA, within 1e-5); `bit_exact` = serial bit-identical correlation."""
    out = {}
    k5 = K - (K % 2)
    fr = ws * n5 * NFRAM
    for tag, prec, fuse in (("", B.PREC_FMA, True), ("bit_exact", B.PREC_EXACT, True), ("unfused_bit_exact", B.PREC_EXACT, False)):
        pw = B.Phasewheel(n5, 1024, FS, device=local); co = B.Stcorrdsp(n5, int(FS), device=local)
        co.set_precision(prec)
        if fuse:
            pw.attach_cor(co)

            def c5(s):
                pw.process_ptr(blk(s), stride, NFRAM)
        else:
            def c5(s):
                co.process_ptr(blk(s), stride, NFRAM)
                pw.process_ptr(blk(s), stride, NFRAM)
        for s in range(W + 1):
            c5(s)
        ms = timed_loop(torch, dist, ws, c5, k5)
        r = {"frames_per_s": fr * k5 / (ms * 1e-3), "ms_per_block": ms / k5, "hbm_frac_per_gpu": fr / ws * 12 * k5 / (ms * 1e-3) / 1e9 / hbm_peak}
        if tag:
            out[tag] = r
        else:
            out.update(r)
            out.update({"stereo_instances_per_gpu": n5, "fused_cor": True, "cor_precision": "B200M_PREC_FMA (time-parallel scan, within 1e-5)",
                        "scaling": "strong" if ws > 1 else "single GPU"})
        del pw, co
    return out


def cpu_baseline(budget_s=8.0, steps=None, warmup=1):
    """The reference's CPU code (oracle/_ref if present, else the port) for the headline workload, on every CPU this process
    may use: persistent pinned workers that own their instances (oracle/cpu_bench.inc).  Also measures one thread alone so
    that the line shows how the host scales (round 1 ran 128 unpinned spawn-per-call threads and got 1.2 M samples/s each)."""
    import _oracle as O
    L = O.load("best")
    kind = L.orc_kind().decode()
    eff, hw, aff, quota = O.cpu_info("best")
    one = O.r128_bench(16, NFRAM, CPU_BLOCKS, 1, steps=8, warmup=1, kind="best")          # ~1 M samples per step: ~1 s
    per_step = N_INST * 2 * NFRAM * CPU_BLOCKS
    if steps is None:
        cal = O.r128_bench(N_INST, NFRAM, CPU_BLOCKS, eff, steps=2, warmup=0, kind="best")
        steps = int(max(3, min(400, budget_s * cal["samples_per_s"] / per_step)))
    full = O.r128_bench(N_INST, NFRAM, CPU_BLOCKS, eff, steps=steps, warmup=warmup, kind="best")
    return {"value": full["samples_per_s"], "unit": "samples/s", "cores": full["threads"], "kind": "reference" if kind == "reference" else "port",
            "sample": "%d of %d stereo instances x %d blocks of %d frames per step, %d steps, %.1f s" % (N_INST, N_INST, CPU_BLOCKS, NFRAM, full["steps"], full["wall_s"]),
            "ms_per_step": full["wall_s"] / full["steps"] * 1e3, "steps": full["steps"],
            "threads": "persistent, one pinned per usable CPU, each owns its instances and input (oracle/cpu_bench.inc)",
            "one_thread_samples_per_s": one["samples_per_s"], "per_thread_samples_per_s": full["per_thread"],
            "scaling_efficiency": full["per_thread"] / one["samples_per_s"], "worker_imbalance": full["imbalance"],
            "hw_threads": hw, "affinity_cpus": aff, "cgroup_quota_cpus": quota or None}


def run_reference(args):
    rank, local, ws = dist_env()
    if rank != 0:
        return
    K, W = args.steps, max(args.warmup, 1)
    cb = cpu_baseline(steps=K, warmup=W)
    out = {"metric": METRIC, "value": cb["value"], "unit": "samples/s", "n_gpus": ws, "steps": K, "warmup": W,
           "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "impl": "reference",
           "config": {"workload": "8192 stereo EBU R128 M+S+I (integrating) + dBTP true-peak 4x (ebur128_run audio cycle), CPU: " + cb["sample"],
                      "block": NFRAM, "fs": FS},
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--headline-only", action="store_true", help="skip the other BASELINE configs, whole-mix and spot check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the headline's last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
