#!/usr/bin/env python
"""Benchmark of the reverse-SDE enhancement hot path (BASELINE.json metric: utterances/sec, 4-s 16 kHz
clips, N=30 predictor-corrector steps = 60 score-network evaluations per utterance).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own enhancement.py path on the host CPU cores (oracle/_ref)

A "step" is one pass of the hot path over one batch of synthetic noisy speech: STFT -> magnitude
compression -> pad -> N-step PC sampling with the NCSN++ score network -> decompression -> iSTFT.
Workload at every N: configs[1] of BASELINE.json (SGMSE+ NCSN++ VoiceBank config, 16 kHz, batch 16 per GPU,
N=30); utterances are independent, so ranks shard the batch with no data-path collective (weak scaling,
NCCL only for the one-off weight broadcast).

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 16000
CLIP_S = 4
# SURVEY.md §8(d): algorithmic work of one NCSN++ forward on one 4-s 16 kHz utterance ([1,4,256,512])
GFLOP_PER_FORWARD = 1064.7


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="utterances per GPU per step")
    ap.add_argument("--micro-batch", type=int, default=16)
    ap.add_argument("--N", type=int, default=30)
    ap.add_argument("--mode", default="fp16_tc")
    ap.add_argument("--lanes", type=int, default=1, help="concurrent launch sequences inside the sampler graph")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json configs[i-1]: 2 = the metric's workload (default, the only one the driver runs); "
                         "3 = ncsnpp_48k 48 kHz batch 8; 4 = dereverb settings N=50 snr=0.33 batch 32 (parity-test cases, "
                         "measurable here for the record; no CPU baseline)")
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=VALUE",
                    help="engine A/B option (Engine.set_option), e.g. --opt pdl=1 with SGMSE_B200_PDL=1; recorded in config")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the enhanced waveforms of the last timed step (float32 [batch, samples]) "
                         "to DIR/enhanced.npy (DIR/enhanced_rank<r>.npy per rank when --gpus > 1); inputs, weights and noise "
                         "seeds are fixed, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 arm computed")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's OWN enhancement.py path on the host cores (oracle/_ref = the unmodified reference package,
# staged by oracle/build_ref.py; falls back to the oracle port, loudly, where it is not staged), bounded sample
# ------------------------------------------------------------------------------------------------
_CPU = {"threads": None, "sweep": None, "forward_s": None, "source": None}


def _thread_candidates():
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    import torch
    cands = {8, 16, 24, 32, 48, 64, avail // 2, avail, torch.get_num_threads()}
    return sorted(c for c in cands if 1 <= c <= avail)


def pick_cpu_threads(forward):
    """Thread sweep on the FULL shape of the workload: one warm + one timed score-network evaluation on a
    [1, 2, 256, 512] input per candidate count, ascending; the fastest wins.  More threads are NOT faster for this
    batch-1 network (MKL-DNN convolutions: 16 threads 3.75 s, 64 threads 5.3 s, 128 threads 73 s per evaluation on the
    128-CPU host of the B200 box, profiles/r02_bench_reference_arm.json), so the sweep stops once two candidates in a row are
    slower than the best so far or one is more than 1.25x slower: the 128-thread point alone would cost 2.5 minutes.  The table goes into the JSON line (`cpu_baseline.thread_sweep_s_per_forward`)."""
    if _CPU["threads"] is not None:
        return _CPU["threads"]
    import torch
    sweep, best, worse = {}, (float("inf"), 1), 0
    for c in _thread_candidates():
        torch.set_num_threads(c)
        forward()
        t0 = time.perf_counter()
        forward()
        dt = time.perf_counter() - t0
        sweep[str(c)] = round(dt, 3)
        if dt < best[0]:
            best, worse = (dt, c), 0
        else:
            worse += 1
            if worse >= 2 or dt > 1.25 * best[0]:      # the curve has turned (3.7 s at 48 threads, 5.1 s at 64, 69 s at 128)
                sweep["stopped_after"] = c
                break
    _CPU.update(threads=best[1], sweep=sweep, forward_s=best[0])
    torch.set_num_threads(best[1])
    return best[1]


def cpu_state():
    """(kind, step_fn): step_fn(n_pc_steps) runs ONE utterance through the enhancement.py:75-96 sequence with an
    n-step PC sampler and returns (seconds total, seconds outside the sampler)."""
    import torch
    from oracle import refshim
    from sgmse_b200.synth import synthetic_speech
    wav = synthetic_speech(1, SR * CLIP_S)
    if refshim.reference_available():
        # BASELINE.md section 3: the reference's own modules, random init (init_scale=1.0), eval(), device='cpu'
        model = refshim.make_score_model("ncsnpp", seed=0)
        from sgmse.util.other import pad_spec
        xprobe = torch.complex(torch.randn(1, 2, 256, 512), torch.randn(1, 2, 256, 512))
        tprobe = torch.tensor([0.5])

        def forward():
            with torch.no_grad():
                model.dnn(xprobe, tprobe)

        def step(n):
            t0 = time.perf_counter()
            y = wav.clone()
            T_orig = y.size(1)                                   # enhancement.py:68
            norm_factor = y.abs().max()                          # :71-72
            y = y / norm_factor
            Y = torch.unsqueeze(model._forward_transform(model._stft(y.to("cpu"))), 0)     # :75
            Y = pad_spec(Y, mode="zero_pad")                     # :76
            sampler = model.get_pc_sampler("reverse_diffusion", "ald", Y.to("cpu"), N=n, corrector_steps=1, snr=0.5)   # :81-82
            t1 = time.perf_counter()
            sample, _ = sampler()                                # :93
            t2 = time.perf_counter()
            x_hat = model.to_audio(sample.squeeze(), T_orig)     # :96
            x_hat = x_hat * norm_factor                          # :99
            x_hat.cpu().numpy()
            t3 = time.perf_counter()
            return t3 - t0, (t1 - t0) + (t3 - t2)
        kind = "reference"
        _CPU["source"] = refshim.reference_kind() + ": " + refshim.REFERENCE_ROOT     # 'staged: .../oracle/_ref' on the GPU box
    else:
        print("bench.py: oracle/_ref is not staged (run __graft_entry__.build() where /root/reference exists): "
              "the CPU arm falls back to the oracle PORT", file=sys.stderr)
        from oracle import weights as o_w, sde as o_sde, spec as o_spec, pipeline as o_pipe, ncsnpp as o_net
        from oracle.arch import NetConfig
        ncfg = NetConfig.ncsnpp()
        sd = o_w.make_state_dict(ncfg, seed=0)
        xprobe = torch.complex(torch.randn(1, 2, 256, 512), torch.randn(1, 2, 256, 512))
        tprobe = torch.tensor([0.5])

        def forward():
            with torch.no_grad():
                o_net.forward(sd, ncfg, xprobe, tprobe)

        def step(n):
            draws = o_sde.make_noise((1, 1, 256, 512), 1 + 2 * n, seed=2000)
            t0 = time.perf_counter()
            o_pipe.enhance(sd, ncfg, o_spec.SpecConfig(), o_sde.OUVE(), wav, draws, N=n)
            return time.perf_counter() - t0, 0.0
        kind = "port"
    pick_cpu_threads(forward)
    return kind, step


def _cpu_line(kind, n_sample, N, ts):
    """ts = [(total seconds, seconds outside the sampler)] of the timed samples."""
    t = sum(a for a, _ in ts) / len(ts)
    tout = sum(b for _, b in ts) / len(ts)
    per_utt = tout + (t - tout) * N / n_sample                  # only the sampler part scales with the number of PC steps
    what = ("the unmodified reference (oracle/_ref: sgmse.model.ScoreModel, enhancement.py:75-96 sequence, device='cpu')"
            if kind == "reference" else "the fp32 torch-CPU oracle PORT (oracle/_ref not staged)")
    return {"value": 1.0 / per_utt, "unit": "utterances/s", "cores": _CPU["threads"], "host_cpus": os.cpu_count(), "kind": kind,
            "sample": f"1 utterance (4 s, 16 kHz) through {what}: STFT + {n_sample} of {N} PC steps ({2 * n_sample} of {2 * N} "
                      f"NCSN++ evaluations) + iSTFT, {t:.1f} s measured per sample ({tout:.2f} s of it outside the sampler); "
                      f"utterances/s = 1 / (outside + sampler x {N}/{n_sample})",
            "reference_source": _CPU.get("source"), "sample_s": round(t, 3), "extrapolated_s_per_utterance": round(per_utt, 2),
            "thread_sweep_s_per_forward": _CPU["sweep"]}, t


def cpu_baseline(n_steps_total=30, n_sample=2):
    kind, step = cpu_state()
    ts = [step(n_sample)]
    return _cpu_line(kind, n_sample, n_steps_total, ts)[0]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, step = cpu_state()
    # bounded sample per step: as many real PC steps as fit ~4 minutes for the whole --steps/--warmup run
    n_warm = max(0, min(args.warmup, 1))
    per_pc_step = 2 * _CPU["forward_s"]
    n_sample = int(max(1, min(args.N, 240.0 / ((args.steps + n_warm) * per_pc_step))))
    for _ in range(n_warm):
        step(n_sample)
    ts = [step(n_sample) for _ in range(args.steps)]
    cb, t = _cpu_line(kind, n_sample, args.N, ts)
    v = cb["value"]
    print(json.dumps({
        "impl": "reference", "metric": "utterances/sec (4 s, 16 kHz, N=30 PC)", "value": v, "unit": "utterances/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # the MEASURED time of one step (= one bounded sample), so that steps x ms_per_step is the real timed region;
        # the whole-utterance figure behind `value` is cpu_baseline.extrapolated_s_per_utterance
        "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args), "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def workload_config(args):
    return {"workload": f"{args.workload_name}, 4-s clips, "
                        f"batch {args.batch} per GPU, PC sampler reverse_diffusion+ald N={args.N} snr {args.snr} "
                        f"({2 * args.N} network evaluations), STFT {args.stft}",
            "baseline_config": args.config,
            "global_batch": args.batch * args.gpus, "per_gpu_batch": args.batch, "micro_batch": args.micro_batch, "lanes": args.lanes,
            "parallelism": f"dp{args.gpus} (batch sharded, no data-path collective)",
            **({"options": list(args.opt)} if getattr(args, "opt", None) else {}),
            "l2": "working set per step (>10 GB of activations per micro-batch) exceeds the 126 MB L2; no flush needed"}


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    from sgmse_b200 import Engine, EngineConfig
    from sgmse_b200.synth import synthetic_blob, synthetic_speech

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ecfg = (EngineConfig.ncsnpp_48k if args.config == 3 else EngineConfig)(mode=args.mode, max_batch=args.micro_batch, use_graphs=True)
    eng = Engine(ecfg, device=dev)
    eng.set_option("lanes", args.lanes)
    for kv in args.opt:
        k, v = kv.split("=")
        eng.set_option(k, int(v))
    # weights: rank 0 creates them, NCCL broadcast over NVLink, packed per rank
    n = eng.weights_numel()
    if rank == 0:
        blob = synthetic_blob(eng, seed=0).to(dev)
    else:
        blob = torch.empty(n, dtype=torch.float32, device=dev)
    if world > 1:
        dist.broadcast(blob, src=0)
    eng.load_blob(blob)
    del blob

    L = SR * CLIP_S
    wav_host = synthetic_speech(args.batch, L, first=rank * args.batch).pin_memory()
    wav_dev = wav_host.to(dev)
    out_dev = torch.empty_like(wav_dev)
    out_host = torch.empty_like(wav_host).pin_memory()
    kw = dict(N=args.N, predictor="reverse_diffusion", corrector="ald", corrector_steps=1, snr=args.snr)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    step_dev = lambda i: eng.enhance(wav_dev, out=out_dev, seed=1 + i, utt_offset=rank * args.batch, **kw)
    step_host = lambda i: eng.enhance(wav_host, out=out_host, seed=1 + i, utt_offset=rank * args.batch, **kw)

    for i in range(args.warmup):
        step_dev(i)
    l0 = eng.counter("kernel_launches")
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms = timed(step_dev, args.steps)
    launches = eng.counter("kernel_launches") - l0
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "enhanced.npy" if world == 1 else f"enhanced_rank{rank}.npy"),
                out_dev.float().cpu().numpy())
    step_host(0)
    ms_e2e = timed(step_host, args.steps)
    clk = clocks.stop() if rank == 0 else None
    assert torch.isfinite(out_dev).all() and torch.isfinite(out_host).all()

    utts = args.batch * world * args.steps
    value = utts / (ms * 1e-3)
    e2e = utts / (ms_e2e * 1e-3)

    roof = None
    if not args.no_roofline and args.mode == "fp16_tc":
        # dominant kernels = the tcgen05 implicit-GEMM convolutions: CUDA events around every launch of one more
        # (eager, un-graphed) step on the launching stream
        eng.set_option("time_convs", 1)
        step_dev(0)
        torch.cuda.synchronize()
        us = eng.counter("timed_conv_tc_us")
        mflop = eng.counter("timed_conv_tc_mflop")
        cnt = eng.counter("timed_conv_tc_count")
        kbytes = eng.counter("timed_conv_tc_kbytes")    # algorithmic bytes of the same launches (inputs once + output once)
        eng.set_option("time_convs", 0)
        pk = peaks()
        ach = mflop / max(us, 1)            # MFLOP/us = TFLOP/s
        # DRAM traffic of the dominant kernel: ncu counters of one launch of the dominant shape, captured from THIS build
        # (tools/make_conv_traffic.py records a digest of the kernel's sources next to the counters); a capture of another
        # build is not reported
        traffic, traffic_note = None, None
        tpath = os.path.join(ROOT, "profiles", "r02_conv_traffic.json")
        if os.path.exists(tpath):
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from make_conv_traffic import source_digest
            tj = json.load(open(tpath))
            if tj.get("source_digest") == source_digest():
                traffic = tj["traffic_bytes_per_launch"]
                traffic_note = {k: tj[k] for k in ("kernel", "shape", "algorithmic_bytes_per_launch", "ratio", "source", "source_digest")}
            else:
                traffic_note = {"stale": f"profiles/r02_conv_traffic.json was captured from kernel sources {tj.get('source_digest')}, "
                                         f"this build is {source_digest()}: re-run tools/make_conv_traffic.py"}
        roof = {"kernel": "tcgen05 implicit-GEMM convolutions (conv_tc6 with fused GroupNorm+SiLU producers; conv_tc4 / conv_tc on the levels below 32 rows)",
                "bound": "tensor", "achieved": round(ach, 1),
                "peak": pk["tflops_sustained"], "unit": "TFLOP/s", "frac": round(ach / pk["tflops_sustained"], 4),
                "traffic": traffic, "traffic_of": traffic_note,
                "launches_timed": cnt, "avg_launch_us": round(us / max(cnt, 1), 1),
                "peak_source": pk["source"] + " (bf16_tflops_sustained: kernel timed inside a long step)",
                "share_of_step": round(us * 1e-3 / (ms / args.steps), 3),
                # the same launches against the other roof: algorithmic HBM bytes / time (KB/us = GB/s)
                "algorithmic_hbm_gbs": round(kbytes / max(us, 1), 1), "hbm_peak_gbs": pk["hbm_gbs"],
                "hbm_frac": round(kbytes / max(us, 1) / pk["hbm_gbs"], 4),
                "algorithmic_gflop_per_step": round(mflop * 1e-3, 1)}
    cb = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(args.N)

    if rank == 0:
        line = {
            "metric": "utterances/sec (4 s, 16 kHz, N=30 PC)" if args.config == 2 else
                      f"utterances/sec (4 s, {SR // 1000} kHz, N={args.N} PC)", "value": round(value, 4), "unit": "utterances/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (fp32 accumulate)" if args.mode != "fp32" else "f32", "data": "synthetic",
            "config": workload_config(args), "rtf": round((ms * 1e-3) / (utts * CLIP_S), 6),
            "e2e": {"value": round(e2e, 4), "unit": "utterances/s", "h2d_bytes_per_step": args.batch * L * 4,
                    "d2h_bytes_per_step": args.batch * L * 4, "ms_per_step": round(ms_e2e / args.steps, 3)},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cb,
            "tflops_effective": round(value * 2 * args.N * GFLOP_PER_FORWARD * 1e-3 / world, 1),
        }
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


WORKLOADS = {
    # name, sampling rate, GFLOP per forward per utterance (SURVEY.md §8d), per-GPU batch, micro-batch, N, snr
    2: dict(name="SGMSE+ NCSN++ (VoiceBank-DEMAND config, 65.6 M params, random init), 16 kHz", sr=16000, gflop=1064.7,
            batch=16, micro=16, N=30, snr=0.5, stft="510/128"),
    3: dict(name="NCSN++ 48 kHz (EARS-WHAM config: backbone ncsnpp_48k, 64.7 M params, random init), 48 kHz", sr=48000,
            gflop=3187.6, batch=8, micro=8, N=30, snr=0.5, stft="1534/384"),
    4: dict(name="SGMSE+ NCSN++ (WSJ0-REVERB dereverberation settings, random init), 16 kHz", sr=16000, gflop=1064.7,
            batch=32, micro=16, N=50, snr=0.33, stft="510/128"),
}


def apply_workload(args):
    """--config 3 / 4 replace the defaults of --batch / --micro-batch / --N (explicit flags still win is NOT attempted:
    a named config means its published settings)."""
    global SR, GFLOP_PER_FORWARD
    w = WORKLOADS[args.config]
    args.snr = w["snr"]
    args.workload_name = w["name"]
    args.stft = w["stft"]
    if args.config != 2:
        args.batch, args.micro_batch, args.N = w["batch"], w["micro"], w["N"]
        args.no_cpu_baseline = True
        SR, GFLOP_PER_FORWARD = w["sr"], w["gflop"]


def main():
    args = parse()
    apply_workload(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
