#!/usr/bin/env python
"""bench.py -- RVC v2/48k inference hot path on B200 (BASELINE.json metric: 48 kHz output samples / s).

One "step" = one 10 s / 16 kHz utterance through the whole path (config #2: v2/48k model, RMVPE f0,
100k-vector IVF2564,Flat index, k=8, index_rate 0.75, x_pad=3 => 16 s of model compute, 479 040 output samples):
high-pass filtfilt + reflect pad -> HuBERT features -> IVF-Flat search + blend || RMVPE f0 -> f0 post-processing ->
SynthesizerTrnMs768NSFsid.infer -> RMS mix + int16.

  value   device-resident: the utterance (float32) already in HBM, CUDA events around the product path's own body
          (Pipeline._dev_body, the very function VC.vc_single runs), replayed as one CUDA graph
  e2e     VC.vc_single (the reference's public entry) with HOST numpy audio in and host int16 audio out:
          pinned H2D of the utterance, the same body, D2H of the int16 result, all host work inside the timed region
  --impl reference   the reference's CPU path (oracle restatement, pinned against the reference's own modules)
                     on the box's host cores for the same metric/config: each step is ONE FULL utterance (all 16 s of model
                     compute), thread count chosen by a short sweep over {8, 16, 32, 64}.
  --impl reference_gpu   SURVEY section 8d(ii): the same PyTorch modules EAGER on this GPU (cuDNN / cuBLAS), fp16 and fp32, with the
                     reference's host round trips preserved (oracle/gpu_ref.py) -- the same-box bar the sm_100a kernels must beat.
Before timing, the default run checks its own output: the product path with the oracle's pitch track and noise draws against the
fp32 CPU oracle's waveform of the same utterance (the cpu_baseline leg computes it anyway): "parity_check" in the JSON line.
Synthetic seeded weights / audio / index (no assets, no network): "data": "synthetic".
  --dump-outputs DIR   after the timed steps, write what the last timed step of each timed path returned as float32 .npy:
                     device_step_audio (the device-resident step's int16 waveform) and vc_single_audio (VC.vc_single's int16
                     waveform).  Weights, audio, index and torch's generator are seeded, so the same arguments give the same
                     inputs on every run and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "retrieval-based-voice-conversion-webui_b200")
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

OUT_SAMPLES = 479040          # 160000 in @16k -> (2*799)*480 - 2*3*48000 out @48k
UTT_SECONDS = 10.0
ALGO_FLOPS = (246.0 + 117.1 + 1833.0) * 1e9     # BASELINE.md section 2, offline fp16-config column


class Cfg:  # the object Pipeline reads (configs/config.py:219-230, fp16 "6G" preset)
    x_pad, x_query, x_center, x_max, is_half = 3, 10, 60, 65, True

    def __init__(self, device):
        self.device = device
        self.rmvpe_state_dict = None


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx, self.samples, self.reasons, self.maxmhz, self.stop_flag = gpu_index, [], set(), 0, False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(", ")
                self.samples.append(float(o[0])); self.maxmhz = float(o[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), o[2:6]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.maxmhz or None,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


WORKLOAD = "configs[1]: v2/48k, RMVPE f0, 100k-vec IVF2564,Flat k=8 rate 0.75, 10s utterance, x_pad=3 (16s compute)"
METRIC = "48kHz audio samples/sec (v2/48k infer, RMVPE, IVF index)"


def make_cpu_pipeline(noise_seed=3):
    from oracle import pipeline as OP, weights as OW
    return OP.OraclePipeline(48000, 3, 10, 60, 65, OW.hubert_weights(777), OW.rmvpe_weights(4321), OW.synth_weights(1234), OW.V2_48K_CONFIG,
                             noise_seed=noise_seed)


def cpu_full_step(pipe, audio, idx):
    """ONE full utterance through the whole reference path on the host (filtfilt, reflect pad, RMVPE f0 + post-processing, HuBERT,
    IVF search + blend, synthesizer, RMS mix, scaling): pipeline.py:186-366 as restated by the oracle."""
    pipe.taps.clear()
    with torch.no_grad():
        return pipe.pipeline(0, audio.copy(), 0, "rmvpe", idx, 0.75, 1, 48000, 0, 0.25, "v2", 0.33)


def pick_cpu_threads(pipe, audio, idx):
    """Thread sweep on a 1.5 s slice of the utterance (the convolutions are small: more threads is not always faster)."""
    from oracle import rmvpe as ORM
    n = os.cpu_count()
    # 128 threads measured 100+ s for this 0.3 s slice on the 128-core box (oversubscribed fork/join on small convolutions): not swept
    cands = sorted({c for c in (8, 16, 32, 64) if c <= n} | {min(n, 16)})
    chunk = np.ascontiguousarray(audio[: 24000])
    res = {}
    for c in cands:
        torch.set_num_threads(c)
        best = 1e9
        for _ in range(2):
            t0 = time.perf_counter()
            with torch.no_grad():
                pitch, pitchf = ORM.calculate(pipe.rw, chunk, 150, 0)
                pipe.vc(torch.tensor([0]), chunk, torch.tensor(pitch).unsqueeze(0).long(), torch.tensor(pitchf.astype(np.float32)).unsqueeze(0),
                        None, None, 0.0, "v2", 0.33)
            best = min(best, time.perf_counter() - t0)
        res[c] = best
    pipe.taps.clear()
    c = min(res, key=res.get)
    torch.set_num_threads(c)
    return c, {str(k): round(v, 3) for k, v in res.items()}


def reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path (oracle restatement) on the host cores, one full utterance per step."""
    if rank != 0:
        return
    from oracle import gpu_ref as GR, ivf as OI, weights as OW
    audio = OW.synth_voice(UTT_SECONDS, seed=0).numpy()
    vec = OW.index_vectors(100000, 768, 0).numpy()
    # faiss is absent: a BLAS-backed IVF search (what faiss-cpu does for nq >= 20) stands in, not the oracle's serial lane-order scan
    idx = GR.BlasIVF(OI.build_ivf(vec, None, seed=0, exact_assign=False))
    idx.ntotal = vec.shape[0]
    idx.reconstruct_n = lambda i0, n: vec[i0:i0 + n]
    pipe = make_cpu_pipeline()
    cores, sweep = pick_cpu_threads(pipe, audio, idx)
    for _ in range(args.warmup):
        cpu_full_step(pipe, audio, idx)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_full_step(pipe, audio, idx)
    dt = time.perf_counter() - t0
    v = args.steps * OUT_SAMPLES / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "rtf_x": v / 48000.0, "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": f"each step = ONE FULL utterance (16 s of model compute, {OUT_SAMPLES} output samples) through the whole reference path; "
                                       f"torch CPU fp32, {cores} threads of {os.cpu_count()} cores (sweep, s per 1.5 s slice: {sweep}); IVF search by BLAS (faiss absent)"},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def reference_gpu_arm(args, rank, world):
    """SURVEY 8d(ii): the oracle's functional PyTorch modules eager on the GPU (cuDNN / cuBLAS), host round trips preserved."""
    if rank != 0:
        return
    from oracle import gpu_ref as GR, ivf as OI, weights as OW
    torch.set_num_threads(min(os.cpu_count(), 32))
    audio = OW.synth_voice(UTT_SECONDS, seed=0).numpy()
    idx = OI.build_ivf(OW.index_vectors(100000, 768, 0).numpy(), None, seed=0, exact_assign=False)
    res = {}
    for half in (True, False):
        g = GR.GpuReference(OW.hubert_weights(777), OW.rmvpe_weights(4321), OW.synth_weights(1234), OW.V2_48K_CONFIG, idx, "cuda:0", half, 3)
        for _ in range(max(args.warmup, 2)):
            g.convert(audio.copy())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            g.convert(audio.copy())
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.steps
        g.convert(audio.copy(), timed=True)
        res["fp16" if half else "fp32"] = {"ms_per_step": dt * 1e3, "samples_per_s": OUT_SAMPLES / dt, "stages_ms": {k: round(v, 2) for k, v in g.stage_ms.items()}}
        del g
        torch.cuda.empty_cache()
    v = res["fp16"]["samples_per_s"]
    line = {"impl": "reference_gpu", "metric": METRIC, "value": v, "unit": "samples/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["fp16"]["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (the reference's is_half GPU default, configs/config.py:38); fp32 alongside", "data": "synthetic",
            "config": {"workload": WORKLOAD}, "variants": res,
            "note": "oracle modules (pinned against the reference's own) eager on the same GPU: cuDNN / cuBLAS kernels, host round trips of "
                    "pipeline.py:118,135-138,172-174 and rmvpe.py:109 preserved, IVF search on the host by BLAS (faiss absent); wall clock, host in -> host out",
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": int(256000 * 4 * 2 + 799 * 768 * 4), "d2h_bytes_per_step": int(1601 * 360 * 4 + 799 * 768 * 4 + 767040 * 4)}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference_gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs is supported with --impl b200 only")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.impl == "reference_gpu":
        reference_gpu_arm(args, rank, world)
        return
    if args.warmup < 3:          # timing hygiene: never fewer than 3 untimed warm-up steps (reported as run)
        args.warmup = 3
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.manual_seed(0)                 # the synthesizer's noise draws: the same on every run
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from rvc_b200 import _lib, synthetic as SY
    from rvc_b200.engine import Index
    from rvc_b200.index_build import build_ivf_layout
    from infer.modules.vc.modules import VC
    from infer.modules.vc.utils import HubertB200
    _lib.init(local_rank)

    # ---- model containers (seeded synthetic checkpoints) ----
    cfg = Cfg(str(dev))
    cfg.rmvpe_state_dict = SY.rmvpe_weights(4321)
    vc = VC(cfg)
    vc.hubert_model = HubertB200(SY.hubert_weights(777), dev)
    cpt = SY.synth_cpt(1234, "v2")
    vc.get_vc(cpt)
    # index: rank 0 builds the layout; the optional one-time broadcast over NCCL shares it (the only collective of the path)
    if rank == 0:
        lay = build_ivf_layout(SY.index_vectors(100000, 768, 0).numpy(), None, seed=0, device=str(dev))
    if world > 1:
        from rvc_b200.dist_utils import broadcast_layout
        lay = broadcast_layout(lay if rank == 0 else None, 0, str(dev))
    index = Index.from_oracle_layout(lay, local_rank)

    audio = SY.synth_voice(UTT_SECONDS, seed=rank).numpy()          # each rank converts its own utterances (weak scaling)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def e2e_step():
        info, out = vc.vc_single(0, audio, 0, None, "rmvpe", index, "", 0.75, 3, 0, 0.25, 0.33)
        assert out is not None, info
        return out[1]

    # ---- device-resident step: the product path's own body (Pipeline._dev_body: filtfilt -> pad -> [RMVPE -> f0 post] ||
    # [HuBERT -> retrieval] -> synthesizer -> RMS mix -> int16) with the utterance already in HBM: same kernels, same stream
    # structure and the same data dependencies (the synthesizer consumes the pitch RMVPE produced in this very step) ----
    pipe = vc.pipeline
    x_dev = torch.from_numpy(np.divide(audio, max(1.0, np.abs(audio).max() / 0.95)).astype(np.float32)).to(dev)
    body_args = (vc.hubert_model, vc.net_g, torch.tensor(0).unsqueeze(0).long(), [0, 0, 0], 0, index, index.vectors, 0.75, 1, 48000,
                 0.25, "v2", 0.33, True)

    def dev_step(use_side=True):
        if use_side:
            return pipe._dev_body(x_dev, *body_args)
        real = pipe._side
        pipe._side = torch.cuda.current_stream()
        try:
            return pipe._dev_body(x_dev, *body_args)
        finally:
            pipe._side = real

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for s, e in ev:
            flush.fill_(1)                      # L2 flush between timed iterations (outside the event pair)
            s.record()
            out = fn()
            e.record()
        torch.cuda.synchronize()
        ms = sum(s.elapsed_time(e) for s, e in ev)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(t.item()), out

    # the device-resident step is a fixed sequence of ~510 launches: capture it once (both streams) and replay the CUDA graph
    for _ in range(2):
        dev_step()
    torch.cuda.synchronize()
    use_graph = os.environ.get("RVCB_BENCH_GRAPH", "1") == "1"
    launches = 0
    step_fn = dev_step
    if use_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            l0 = _lib.lib().rvcb_launch_count()
            with torch.cuda.graph(graph):
                graph_out = dev_step()
            launches = _lib.lib().rvcb_launch_count() - l0
            step_fn = graph.replay
        except Exception as e:      # capture is an optimisation of launch overhead only; report and fall back to eager launches
            print(f"[bench] CUDA graph capture failed ({e}); timing eager launches", file=sys.stderr)
            use_graph = False
            torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = _lib.lib().rvcb_launch_count()
    dev_ms, dev_out = timed(step_fn, args.steps, args.warmup)
    if not use_graph:
        launches = (_lib.lib().rvcb_launch_count() - l0) // (args.steps + args.warmup)
    # copied before vc_single runs: its graphs share the model handles with the device-resident step
    dev_out = (graph_out if use_graph else dev_out).float().cpu().numpy()
    e2e_ms, e2e_out = timed(e2e_step, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "device_step_audio.npy"), dev_out)
        np.save(os.path.join(args.dump_outputs, "vc_single_audio.npy"), np.asarray(e2e_out, dtype=np.float32))
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- the same step with the synthesizer decoding EVERY frame (RVCB_TRIM=0), i.e. without restricting the flow / decoder to the
    # frames the caller keeps (the x_pad context is discarded at pipeline.py:295); the kept samples are bit-identical either way ----
    full_decode = None
    if use_graph:
        try:
            os.environ["RVCB_TRIM"] = "0"
            for _ in range(2):
                dev_step()
            torch.cuda.synchronize()
            g_full = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_full):
                out_full = dev_step()
            fms, _ = timed(g_full.replay, args.steps, args.warmup)
            graph.replay()
            torch.cuda.synchronize()
            same = bool(torch.equal(out_full, graph_out)) if (out_full.dtype == graph_out.dtype and out_full.shape == graph_out.shape) else None
            full_decode = {"ms_per_step": fms / args.steps, "value": world * args.steps * OUT_SAMPLES / (fms * 1e-3), "unit": "samples/s",
                           "what": "RVCB_TRIM=0: flow + decoder over all 1598 frames incl. the 2 x 3 s of x_pad context that pipeline.py:295 discards",
                           "int16_output_identical_to_trimmed_step": same,
                           "note": "noise is drawn inside each graph, so the two int16 outputs are only compared when the draws coincide; "
                                   "tests/test_synth_gpu.py proves bit-equality of the kept samples on shared noise"}
        except Exception as e:
            full_decode = {"error": str(e)}
            torch.cuda.synchronize()
        finally:
            os.environ.pop("RVCB_TRIM", None)

    # ---- throughput mode: several utterances in flight on one GPU (batch conversion, BASELINE config #4's per-GPU work): every
    # utterance is its own captured graph over its own handles (arenas are per handle) replayed on its own stream; a single
    # utterance is latency-bound (two branches of ~200 small launches), so independent utterances fill the idle SMs ----
    conc_levels = sorted({int(c) for c in os.environ.get("RVCB_BENCH_CONC", "2,4").split(",") if c.strip() and int(c) > 1})
    conc_res = None
    if use_graph and conc_levels:
        try:
            graphs, keep = [graph], []
            for i in range(1, max(conc_levels)):
                vc2 = VC(cfg)
                vc2.hubert_model = HubertB200(SY.hubert_weights(777), dev)
                vc2.get_vc(SY.synth_cpt(1234, "v2"))
                idx2 = Index.from_oracle_layout(lay, local_rank)
                a2 = SY.synth_voice(UTT_SECONDS, seed=100 + 10 * rank + i).numpy()
                x2 = torch.from_numpy(np.divide(a2, max(1.0, np.abs(a2).max() / 0.95)).astype(np.float32)).to(dev)
                args2 = (vc2.hubert_model, vc2.net_g, torch.tensor(0).unsqueeze(0).long(), [0, 0, 0], 0, idx2, idx2.vectors, 0.75, 1, 48000,
                         0.25, "v2", 0.33, True)
                for _ in range(2):
                    vc2.pipeline._dev_body(x2, *args2)
                torch.cuda.synchronize()
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2):
                    o2 = vc2.pipeline._dev_body(x2, *args2)
                graphs.append(g2)
                keep.append((vc2, idx2, x2, args2, o2))
            cstreams = [torch.cuda.Stream(device=dev) for _ in graphs]

            def conc_step(n):
                cur = torch.cuda.current_stream()
                ev0 = torch.cuda.Event()
                ev0.record(cur)
                for st_, g_ in zip(cstreams[:n], graphs[:n]):
                    st_.wait_event(ev0)
                    with torch.cuda.stream(st_):
                        g_.replay()
                    e_ = torch.cuda.Event()
                    e_.record(st_)
                    cur.wait_event(e_)
            sweep = {}
            for n in conc_levels:
                cms, _ = timed(lambda: conc_step(n), args.steps, args.warmup)
                sweep[n] = {"ms_per_step": cms / args.steps, "ms_per_utterance": cms / args.steps / n,
                            "value": world * n * args.steps * OUT_SAMPLES / (cms * 1e-3)}
            best = min(sweep, key=lambda n: sweep[n]["ms_per_utterance"])
            conc_res = {"utterances_in_flight": best, "ms_per_step": sweep[best]["ms_per_step"], "value": sweep[best]["value"],
                        "unit": "samples/s", "by_utterances_in_flight": {str(n): sweep[n] for n in sweep},
                        "what": "n independent 10 s utterances per step, one captured graph + stream + handle set each, device-resident "
                                "(what VC.vc_multi's RVCB_LANES does); 1 in flight = the headline step"}
            del keep
        except Exception as e:
            conc_res = {"error": str(e)}
            torch.cuda.synchronize()

    # ---- BASELINE config #3 (realtime gui.py block: 160 ms at 48 kHz, extra 2.5 s, crossfade 0.05 s): per-block latency of
    # rtrvc.RVC.infer + the device-side callback tail (envelope mix + SOLA, gui.py:1024-1087) + D2H of the output block ----
    realtime = None
    if world == 1:
        from infer.lib.rtrvc import RVC
        from infer.modules.gui import RealtimeTail
        tail = RealtimeTail(48000, 0.16, 0.05, 2.5, str(dev))
        rt = RVC(0, 0, SY.synth_cpt(1234, "v2"), index, 0.75, device=str(dev), hubert_model=vc.hubert_model, rmvpe_state_dict=cfg.rmvpe_state_dict)
        nblk, nwarm = 300, 20
        stream16 = SY.synth_voice(2.72 + 0.16 * (nblk + nwarm) + 0.1, seed=5).to(dev)
        inp48 = SY.synth_voice(0.25, sr=48000, seed=6).to(dev)
        lat = []
        for b in range(nblk + nwarm):
            win = stream16[b * tail.block_frame_16k: b * tail.block_frame_16k + tail.input_frames_16k]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            y = rt.infer(win, tail.block_frame_16k, tail.skip_head, tail.return_length, "rmvpe")
            out_blk = tail.process(y, inp48, 0.0)            # gui.py default rms_mix_rate 0 -> envelope mix on
            out_blk.cpu()                                    # the callback copies the block to the output ring (gui.py:1088-1094)
            lat.append((time.perf_counter() - t0) * 1e3)
        lat = np.array(lat[nwarm:])
        realtime = {"config": "configs[2]: 160 ms blocks, 43520-sample 16 kHz window, skip_head 250, return_length 21, v2/48k + RMVPE + 100k index",
                    "blocks": int(nblk), "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)), "max_ms": float(lat.max()),
                    "block_period_ms": 160.0, "what": "rtrvc.RVC.infer + RealtimeTail.process (envelope mix + SOLA) + D2H of the 7680-sample block, wall clock"}
        # the whole callback as one object: host block in -> host block out (gui.py:940-1090), one H2D + one graph + one D2H
        try:
            from infer.modules.gui import RealtimeBlock
            mic = SY.synth_voice(0.16 * (nblk + nwarm) + 0.1, sr=48000, seed=7).numpy()

            def callback_latency(**kw):
                blk = RealtimeBlock(rt, samplerate=48000, block_time=0.16, crossfade_time=0.05, extra_time=2.5, device=str(dev), **kw)
                ls = []
                for b in range(nblk + nwarm):
                    ind = mic[b * blk.block_frame: (b + 1) * blk.block_frame]
                    t0 = time.perf_counter()
                    blk.process(ind)
                    ls.append((time.perf_counter() - t0) * 1e3)
                ls = np.array(ls[nwarm:])
                return {"p50_ms": float(np.percentile(ls, 50)), "p99_ms": float(np.percentile(ls, 99)), "max_ms": float(ls.max())}
            realtime["callback"] = {
                "what": "RealtimeBlock.process: host numpy block in -> host numpy block out (input ring, 48k->16k resampler, RVC.infer, "
                        "envelope mix, SOLA as ONE CUDA graph + H2D + D2H), wall clock",
                "gui_defaults": callback_latency(rms_mix_rate=0.0),
                "with_input_and_output_noise_gate": callback_latency(rms_mix_rate=0.0, I_noise_reduce=True, O_noise_reduce=True)}
        except Exception as e:
            realtime["callback"] = {"error": repr(e)[:300]}
            torch.cuda.synchronize()
        del rt, tail

    # ---- roofline of the dominant kernel family (gemm_tc): live CUDA events around every launch of one step set ----
    import ctypes as C
    _lib.check(_lib.lib().rvcb_prof_begin())
    for _ in range(3):
        dev_step(use_side=False)      # serial, so every launch's event pair times that kernel alone
    gms, gn = C.c_double(0), C.c_ulonglong(0)
    _lib.check(_lib.lib().rvcb_prof_end(C.byref(gms), C.byref(gn)))
    gemm_ms_per_step = gms.value / 3
    cls = [(C.c_double * 3)() for _ in range(4)]
    _lib.check(_lib.lib().rvcb_prof_classes(*cls))
    ws_ms, ws_n, ws_flops, ws_bytes = cls[0][1] / 3, cls[1][1] / 3, cls[2][1] / 3, cls[3][1] / 3
    fu_ms, fu_n, fu_flops, fu_bytes = cls[0][2] / 3, cls[1][2] / 3, cls[2][2] / 3, cls[3][2] / 3
    pk, pk_src = peaks()
    exec_flops = (cls[2][0] + cls[2][1] + cls[2][2]) / 3          # executed 2*M*N*K of every tcgen05 launch (incl. K padding), per step
    achieved = exec_flops / (gemm_ms_per_step * 1e-3) / 1e12
    peak = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
    voc_ms, voc_flops = fu_ms + ws_ms, fu_flops + ws_flops

    value = world * args.steps * OUT_SAMPLES / (dev_ms * 1e-3)
    e2e_v = world * args.steps * OUT_SAMPLES / (e2e_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate+residuals",
        "data": "synthetic", "rtf_x_per_gpu": value / world / 48000.0,
        "config": {"workload": WORKLOAD},
        "decoder_trim": "flow / decoder run over the kept frames + receptive-field margins (1030 + 80 of 1598 frames); kept samples bit-identical "
                        "to the full decode (rvcb_synth_infer_keep, tests/test_synth_gpu.py); 'full_decode' times the untrimmed step",
        "timing": {"l2": "256 MiB flush between timed iterations", "utterances_per_gpu_per_step": 1,
                   "device_step": f"CUDA graph replay of the {int(launches)}-launch step" if use_graph else "eager launches"},
        "e2e": {"value": e2e_v, "unit": "samples/s", "h2d_bytes_per_step": int(160000 * 4 + 8),   # the utterance (float32, one pinned copy) + speaker id
                "d2h_bytes_per_step": int(OUT_SAMPLES * 2),  # mixed + normalised waveform, int16
                "ms_per_step": e2e_ms / args.steps, "rtf_x_per_gpu": e2e_v / world / 48000.0,
                "api": "infer.modules.vc.VC.vc_single (host numpy in, host int16 out)"},
        "gpu_launches": int(launches * args.steps),
        "gpu_launches_per_step": int(launches),
        "clocks": sampler.summary(),
        "realtime": realtime,
        "throughput_concurrent": conc_res,
        "full_decode": full_decode,
        # dominant kernel by work: the vocoder's residual-block convolutions (stages 2-3: one fused launch per residual block,
        # resblock_fused_kernel; 27 % of the utterance's FLOPs).  Tensor-bound by design: x in / y out are the only HBM traffic.
        "roofline": {"bound": "tensor", "achieved": fu_flops / max(fu_ms, 1e-9) / 1e9, "peak": peak, "unit": "TFLOP/s",
                     "frac": fu_flops / max(fu_ms, 1e-9) / 1e9 / peak,
                     "traffic": 147.3e6, "traffic_note": "dram read+write of one fused launch (ncu --set full, profiles/prof_r2c_rb64_metrics.txt: 98.8 MB read + 48.5 MB written) "
                                                         "vs 196 MB algorithmic (x in + y out, fp32): part of y is still in the 126 MB L2 when the kernel ends",
                     "kernel": "resblock_fused_kernel<C, NB, EW, MINB, RES> (one launch per ResBlock1 of vocoder stages 2-3: 6 convolutions, residual stream in TMEM)",
                     "launches_per_step": fu_n, "avg_launch_us": fu_ms / max(fu_n, 1) * 1e3, "algorithmic_flops_per_step": fu_flops,
                     "algorithmic_bytes_per_step": fu_bytes, "hbm_view_gbs": fu_bytes / max(fu_ms, 1e-9) / 1e6, "peak_source": pk_src,
                     "limiter": "shared-memory operand reads of SS-mode tcgen05.mma at N = C_out <= 64 (4 KB of A per M=128,K=16 step: ~46 / 60 cycles per MMA "
                                "at N = 32 / 64 instead of 16 / 32) and the 64 B/clk TMEM read of the on-chip epilogue steps (RVCB_RB_TRACE, DESIGN.md)"},
        "roofline_ws": {"bound": "hbm", "achieved": ws_bytes / max(ws_ms, 1e-9) / 1e6, "peak": pk.get("hbm_gbs"), "unit": "GB/s",
                        "frac": ws_bytes / max(ws_ms, 1e-9) / 1e6 / pk.get("hbm_gbs"),
                        "kernel": "gemm_ws2_kernel<*> / gemm_ws_kernel<*> (layer-by-layer weight-stationary convolutions: vocoder stage 1, C = 128)",
                        "launches_per_step": ws_n, "algorithmic_bytes_per_step": ws_bytes,
                        "tensor_view": {"achieved_tflops": ws_flops / max(ws_ms, 1e-9) / 1e9, "frac_of_bf16_sustained": ws_flops / max(ws_ms, 1e-9) / 1e9 / peak}},
        "roofline_vocoder_resblocks": {"bound": "tensor", "achieved": voc_flops / max(voc_ms, 1e-9) / 1e9, "peak": peak, "unit": "TFLOP/s",
                                       "frac": voc_flops / max(voc_ms, 1e-9) / 1e9 / peak, "ms_per_step": voc_ms,
                                       "hbm_bytes_per_step": fu_bytes + ws_bytes, "kernel": "fused + weight-stationary families together (stages 1-3)"},
        "roofline_all_gemm": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "traffic": None, "kernel": "every tcgen05 launch of one utterance (gemm_tc / gemm_sk / gemm_ws* / resblock_fused), timed serially",
                     "launches_per_step": int(gn.value // 3), "ms_per_step": gemm_ms_per_step, "peak_source": pk_src,
                     "executed_flops_per_step": exec_flops, "nominal_flops_full_decode": ALGO_FLOPS},
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # (1) e2e through the reference's literal call: wav FILE path in, .index FILE path in (pipeline.py:213-215 re-reads the
        #     index file on every call; here it is parsed once and cached by (path, mtime)), cache warm
        import tempfile
        from scipy.io import wavfile
        from rvc_b200 import faiss_io
        with tempfile.TemporaryDirectory() as td:
            wpath, ipath = os.path.join(td, "utt.wav"), os.path.join(td, "added_IVF2564_Flat_nprobe_1_bench_v2.index")
            wavfile.write(wpath, 16000, audio.astype(np.float32))
            faiss_io.write_index(ipath, lay)
            def file_step():
                info, out = vc.vc_single(0, wpath, 0, None, "rmvpe", ipath, "", 0.75, 3, 0, 0.25, 0.33)
                assert out is not None, info
            for _ in range(3):
                file_step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                file_step()
            line["e2e"]["file_paths_ms_per_step"] = (time.perf_counter() - t0) / 5 * 1e3
            line["e2e"]["file_paths_note"] = "vc_single(sid, wav path, ..., .index path): wav decode + the same body + int16 out, index cache warm"
        # (2) CPU baseline: ONE FULL utterance through the oracle pipeline on the host cores (threads by sweep, warm), and the
        #     self-check: the product path with the oracle's pitch track and noise draws against that very waveform
        from oracle import ivf as OI
        assign = np.empty(lay.vectors.shape[0], dtype=np.int64)
        for l in range(len(lay.list_off) - 1):
            assign[lay.list_ids[lay.list_off[l]:lay.list_off[l + 1]]] = l
        oidx = OI.IVFFlat(lay.centroids, lay.vectors, assign)
        cpipe = make_cpu_pipeline()
        cpu_threads, sweep = pick_cpu_threads(cpipe, audio, oidx)
        t0 = time.perf_counter()
        ref = cpu_full_step(cpipe, audio, oidx)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": OUT_SAMPLES / dt, "unit": "samples/s", "cores": cpu_threads, "kind": "port",
                                "sample": f"ONE FULL utterance (16 s of model compute, {OUT_SAMPLES} output samples) through the whole reference path, after a "
                                          f"warm-up slice; torch CPU fp32, {cpu_threads} threads of {os.cpu_count()} cores (sweep, s per 1.5 s slice: {sweep}); "
                                          "IVF search by the oracle's exact lane-order scan (the --impl reference arm uses BLAS)"}
        tap = cpipe.taps[0]
        vc.net_g.set_noise(*tap["noise"])
        got = pipe.pipeline(vc.hubert_model, vc.net_g, 0, audio.copy(), [0, 0, 0], 0, (cpipe.pitch[0].numpy(), cpipe.pitchf[0].numpy().astype(np.float64)),
                            index, 0.75, 2, 3, 48000, 0, 0.25, "v2", 0.33)
        err = float(np.abs(got - ref).max() / 32768.0)
        line["parity_check"] = {"max_abs_err_fullscale": err, "bound": 1.5e-3, "ok": bool(err <= 1.5e-3), "samples": int(ref.shape[0]),
                                "what": "Pipeline.pipeline on the bench utterance with the oracle's pitch track + noise draws vs the fp32 CPU oracle waveform "
                                        "(north_star 1e-3; the reference's own fp16 GPU path measures 2.0e-3, profiles/r2a_parity_config2.json)"}
        assert err <= 1.5e-3, f"bench self-check failed: end-to-end max abs err {err}"
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
