#!/usr/bin/env python
"""Benchmark of the MASR inference hot path (BASELINE.json): audio-seconds per second for
fbank -> Conformer encoder -> CTC greedy on `conformer_streaming_fbank`, batch 32 x 10 s @ 16 kHz
per GPU (weak scaling: every rank owns 32 utterances; token ids are gathered over NCCL).

    python bench.py --gpus 1 --steps 10 --warmup 3            # CUDA path (the product)
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy
    python bench.py --impl reference --steps 2 --warmup 1      # reference CPU arm (oracle port) on host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \\
           bench.py --gpus N --steps K --warmup W

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the meaning of every key.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SAMPLE_RATE = 16000
UTT_SAMPLES = 160000           # 10 s
BATCH_PER_GPU = 32
VOCAB = 4233
WORKLOAD = "conformer.yml streaming=True (causal), full-context predict, 32x10s 16kHz per GPU, ctc_greedy, V=4233"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self._halt = threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def make_waves(rank, n=BATCH_PER_GPU):
    from masr_b200 import synth
    return [synth.noise_audio(1000 * rank + i, UTT_SAMPLES) for i in range(n)]


def dump_outputs(out_dir, ws):
    """Write what a caller of the timed step receives, from its packed outputs ``ws``, as DIR/<name>.npy: token ids
    [B, T] (-1 past each utterance's token count), token counts, greedy scores (0..100) and front-end status flags."""
    from masr_b200.engine import greedy_score
    tok = ws["tokens"].cpu().numpy()
    ntok = ws["ntok"].cpu().numpy()
    psum, pcount = ws["psum"].cpu().numpy(), ws["pcount"].cpu().numpy()
    arrays = {"token_ids": np.where(np.arange(tok.shape[1]) < ntok[:, None], tok, -1).astype(np.float32),
              "token_counts": ntok.astype(np.float32),
              "scores": np.array([greedy_score(s, c) for s, c in zip(psum, pcount)], np.float64),
              "status": ws["status"].cpu().numpy().astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
def cpu_reference_pass(sd, cfg, waves, vocab):
    """The reference's own CPU path, restated (oracle port): per utterance featurize -> get_encoder_out ->
    greedy_decoder, exactly the loop `MASRPredictor.predict` runs (B=1 API)."""
    from oracle import conformer as oc, ctc as octc, fbank as ob
    out = []
    with torch.no_grad():
        for w in waves:
            feat = torch.from_numpy(ob.featurize(w.copy()))
            probs = oc.get_encoder_out(sd, cfg, feat[None])[0].numpy()
            out.append(octc.greedy_decode(probs, vocab))
    return out


def best_cpu_threads(sd, cfg, one_wave, vocab):
    """The reference leaves torch's intra-op thread count at its default (= all cores), which is far from
    optimal for B=1 on a many-core host; give the CPU arm its best case: try a few thread counts on one
    utterance and keep the fastest.  Returns the thread count left set."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (4, 8, 16, 32, avail) if c <= avail})
    best, best_t = cands[0], float("inf")
    probe = [one_wave[0][:48000]]                 # 3 s probe keeps the search to a few seconds
    for c in cands:
        torch.set_num_threads(c)
        cpu_reference_pass(sd, cfg, probe, vocab)
        t0 = time.perf_counter()
        cpu_reference_pass(sd, cfg, probe, vocab)
        dt = time.perf_counter() - t0
        if dt > 4 * best_t:
            break
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def run_reference(args):
    """`--impl reference`: the oracle port on the host cores.  Rank 0 only; each step is a bounded
    sample (SAMPLE utterances of the 32 x 10 s batch)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from masr_b200 import synth
    from oracle import conformer as oc, ref_shims
    sample = args.ref_sample
    waves = make_waves(0, sample)
    kind = "port"
    if ref_shims.reference_available() and os.environ.get("MASR_REFERENCE_ARM", "auto") != "port":
        # a reference tree is present (build container): time the UNMODIFIED masr.predict.MASRPredictor.predict loop
        import tempfile
        kind = "reference"
        pred = ref_shims.build_real_predictor(tempfile.mkdtemp(prefix="masr_ref_arm_"), True, 0, VOCAB)
        cores = torch.get_num_threads()

        def one_pass(ws):
            return [pred.predict(audio_data=w.copy()) for w in ws]
    else:
        sd = synth.to_torch(synth.conformer_state_dict(0, VOCAB))
        cfg = oc.ConformerConfig()
        vocab = synth.vocabulary(VOCAB)
        cores = best_cpu_threads(sd, cfg, waves[:1], vocab)

        def one_pass(ws):
            return cpu_reference_pass(sd, cfg, ws, vocab)
    for _ in range(args.warmup):
        one_pass(waves[:1])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass(waves)
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    audio_s = sample * UTT_SAMPLES / SAMPLE_RATE
    v = audio_s / dt
    line = {"impl": "reference", "metric": "audio_seconds_per_second", "value": v, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": f"{sample} of 32 utterances per step, B=1 loop"},
            "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": cores, "kind": kind,
                             "sample": f"{sample} x 10 s utterances per step, {args.steps} steps, torch CPU threads={cores}"
                                       + (" (best of 4..all)" if kind == "port" else " (the reference's default: all cores); unmodified masr.predict.MASRPredictor.predict")},
            "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-sample", type=int, default=4, help="utterances per step of the reference CPU arm")
    ap.add_argument("--cpu-baseline-utts", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0's utterances) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
        return
    if args.warmup < 3:
        args.warmup = 3                      # timing rule: W >= 3

    import faulthandler
    import torch.distributed as dist
    from masr_b200 import _lib, synth
    # a hung collective must not eat the GPU budget: dump every thread's stack and exit if the run stalls
    faulthandler.dump_traceback_later(int(os.environ.get("MASR_BENCH_WATCHDOG_S", "420")), exit=True)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.load()                               # built in place by __graft_entry__.build(); nothing is compiled here
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None
    if world > 1 and os.environ.get("MASR_BENCH_AFFINITY", "1") != "0":
        # one process per GPU: keep this rank's staging threads and its pinned buffers on the CPUs / NUMA node next to ITS GPU
        # (8 ranks x (4 stager threads + 20 MB pinned memcpy per step) otherwise contend across sockets: e2e efficiency 0.91 at N=8 in r01)
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
            ncpu = os.cpu_count() or 1
            masks = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
            cpus = {64 * i + b for i, m in enumerate(masks) for b in range(64) if (m >> b) & 1}
            cpus &= set(os.sched_getaffinity(0))
            if cpus:
                os.sched_setaffinity(0, cpus)
                numa = f"{len(cpus)} GPU-local CPUs"
        except Exception as e:                      # best effort: no NVML / no permission -> default placement
            numa = f"unavailable ({type(e).__name__})"
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")       # whatever NCCL logs must not land on stdout
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sdn = synth.conformer_state_dict(0, VOCAB)
    # the user-facing object: the MASRPredictor drop-in, built from the reference's file formats
    import tempfile
    from masr_b200.predict import MASRPredictor
    tmp = tempfile.mkdtemp(prefix=f"masr_b200_bench_r{rank}_")
    mp, vp = os.path.join(tmp, "inference.pt"), os.path.join(tmp, "vocabulary.txt")
    torch.save(synth.to_torch(sdn), mp)
    synth.write_vocabulary(vp, VOCAB)
    cfg = {"use_model": "conformer", "streaming": True, "decoder": "ctc_greedy",
           "preprocess_conf": {"feature_method": "fbank", "n_mels": 80, "sample_rate": 16000, "use_dB_normalization": True,
                               "target_dB": -20},
           "dataset_conf": {"dataset_vocab": vp}}
    pred = MASRPredictor(configs=cfg, model_path=mp, use_gpu=True)
    eng = pred.predictor
    os.remove(mp)
    waves = make_waves(rank)
    audio_s_rank = BATCH_PER_GPU * UTT_SAMPLES / SAMPLE_RATE
    lengths = [UTT_SAMPLES] * BATCH_PER_GPU
    offs = torch.tensor(np.arange(BATCH_PER_GPU + 1, dtype=np.int64) * UTT_SAMPLES, device=dev)
    wave_dev = torch.from_numpy(np.concatenate(waves)).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    T = 248
    gather_state = {}

    def gather_pack(ws):
        """The only collective of the path: every rank's packed outputs (token ids | counts | status | score sums: one int32
        buffer, 33 KB) -> all ranks, one NCCL all_gather_into_tensor over NVLink.  Called INSIDE the CUDA-graph capture of the
        device step (engine.graph_tail_hook), so a graph replay enqueues the whole step incl. the collective."""
        pack = ws["out_pack"]
        n = pack.numel()
        buf = gather_state.get(("gbuf", n))
        if buf is None:
            buf = gather_state[("gbuf", n)] = torch.zeros(world * n, dtype=pack.dtype, device=pack.device)
        dist.all_gather_into_tensor(buf, pack)
        return buf

    graph_gather = False
    if world > 1:
        dist.all_gather_into_tensor(torch.zeros(world * 8, dtype=torch.int32, device=dev), torch.zeros(8, dtype=torch.int32, device=dev))
        torch.cuda.synchronize(dev)                  # communicator + channels are up before any capture
        if eng.use_graphs and os.environ.get("MASR_GRAPH_GATHER", "1") != "0":
            eng.graph_tail_hook = gather_pack
            graph_gather = True
    try:
        resident = eng.prepare_resident(waves) if eng.use_graphs else None
    except Exception as e:                            # NCCL refused the capture: fall back to an eager collective after the replay
        if not graph_gather:
            raise
        sys.stderr.write(f"[bench] capturing the all-gather failed ({type(e).__name__}: {e}); eager collective instead\n")
        eng.graph_tail_hook, graph_gather = None, False
        eng._graphs.clear()
        resident = eng.prepare_resident(waves)

    def device_step(eager=False, gather=True):
        """One pass of the hot path with inputs resident in HBM: fbank -> encoder -> CTC greedy
        (+ the token gather across ranks).  Replayed as one CUDA graph; `eager` = the same kernels launched one
        by one (used for the per-kernel event timing of the roofline leg)."""
        if resident is not None and not eager:
            ws = resident()
            if world > 1 and gather and not graph_gather:
                gather_pack(ws)
        else:
            hook, eng.graph_tail_hook = eng.graph_tail_hook, None
            feats, frames, status = eng.fbank(None, True, -20.0, wave_dev=wave_dev, offsets_dev=offs, lengths=lengths)
            enc, tl, Tm, ws = eng.encode(feats, frames)
            eng.ctc_greedy(enc, tl, Tm, ws)
            eng.graph_tail_hook = hook
            if world > 1 and gather:
                gather_pack(ws)
        return ws

    def solo_tokens(ws_list):
        """Token ids of a batch computed by THIS rank alone, eagerly (the captured step contains a collective)."""
        ug, eng.use_graphs = eng.use_graphs, False
        try:
            return eng.transcribe(ws_list).tokens
        finally:
            eng.use_graphs = ug

    def unpack(buf, r, B, Tt):
        """rank r's slice of a gathered pack -> (token lists, counts)."""
        n = B * Tt + 4 * B
        on = buf[r * n:(r + 1) * n].cpu().numpy()
        tok, ntok = on[:B * Tt].reshape(B, Tt), on[B * Tt:B * Tt + B]
        return [tok[b, :ntok[b]].tolist() for b in range(B)]

    for _ in range(args.warmup):
        device_step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = eng.launches
    evs = []
    barrier()
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()                         # L2 flush between timed iterations (outside the event bracket)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ws_last = device_step()
        e1.record()
        evs.append((e0, e1))
    barrier()
    wall = time.perf_counter() - wall0
    launches = (eng.launches - launches0) // max(1, args.steps)
    dev_ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    value = world * audio_s_rank / (dev_ms * 1e-3)

    clocks = sampler.stop() if sampler else None      # clocks are sampled over the device-timed region only
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ws_last)      # before any later leg replays the same graph buffers

    # ---- the gathered result is checked on hardware: rank 0 recomputes OTHER ranks' shards and compares the token ids ----
    gather_verified = None
    strong = None
    if world > 1:
        ws = device_step()
        torch.cuda.synchronize(dev)
        Tt = ws["tokens"].shape[1]
        gbuf = gather_state[("gbuf", ws["out_pack"].numel())]
        if rank == 0:
            ok = unpack(gbuf, 0, BATCH_PER_GPU, Tt) == solo_tokens(waves)
            for r in sorted({1, world - 1}):
                ok = ok and unpack(gbuf, r, BATCH_PER_GPU, Tt) == solo_tokens(make_waves(r))
            gather_verified = bool(ok)
        barrier()
        # ---- strong scaling (SURVEY 8d/8e): ONE 32-utterance batch owned by rank 0, scattered over NCCL inside the timed
        #      region (32/N utterances per GPU), decoded, gathered back; checked against rank 0's own full-batch result ----
        if BATCH_PER_GPU % world == 0 and eng.use_graphs:
            Bs = BATCH_PER_GPU // world
            batch0 = make_waves(0)
            full_tokens = solo_tokens(batch0) if rank == 0 else None
            res_s = eng.prepare_resident(batch0[rank * Bs:(rank + 1) * Bs])
            recv = res_s.g["wave"][:Bs * UTT_SAMPLES]
            all_dev = torch.from_numpy(np.concatenate(batch0)).to(dev) if rank == 0 else None
            chunks = list(all_dev.view(world, Bs * UTT_SAMPLES)) if rank == 0 else None

            def strong_step():
                dist.scatter(recv, scatter_list=chunks, src=0)
                w_ = res_s()
                if not graph_gather:
                    gather_pack(w_)
                return w_
            for _ in range(3):
                strong_step()
            barrier()
            sev = []
            for _ in range(args.steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                w_ = strong_step()
                e1.record()
                sev.append((e0, e1))
            barrier()
            ms = sum(a.elapsed_time(b) for a, b in sev) / args.steps
            tt = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
            if rank == 0:
                Tts = w_["tokens"].shape[1]
                sbuf = gather_state[("gbuf", w_["out_pack"].numel())]
                got = [t for r in range(world) for t in unpack(sbuf, r, Bs, Tts)]
                strong = {"value": BATCH_PER_GPU * UTT_SAMPLES / SAMPLE_RATE / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms,
                          "global_batch": BATCH_PER_GPU, "per_gpu_batch": Bs,
                          "path": "rank 0 owns the batch in HBM -> NCCL scatter -> per-rank CUDA-graph step -> NCCL all-gather of the packed ids",
                          "ids_match_single_gpu": bool(got == full_tokens)}
            barrier()

    # ---- end to end through the public API: host float32 buffers in, token ids + score out --------------
    # (1) synchronous calls: predict_batch(batch) returns before the next batch is touched
    for _ in range(2):
        pred.predict_batch(waves)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = pred.predict_batch(waves)
    torch.cuda.synchronize(dev)
    sync_s = (time.perf_counter() - t0) / args.steps
    # (2) the throughput API: predict_batches(stream of batches) stages batch k+1 (pinned pack + H2D on a copy stream)
    #     while batch k computes; every step still copies its 20 MB of host samples in and its ids/scores out
    # N > 1: every rank pipelines its own shard; the one collective of the path (token ids + counters of every rank's
    # shard, NCCL all-gather of the packed int32 outputs) is enqueued on the device right after each step
    hook = None
    if world > 1:
        def hook(pack):
            if graph_gather:
                return                                # the all-gather is part of the captured step
            n = pack.numel()
            if gather_state.get("e2e_n") != n:
                gather_state["e2e_buf"] = torch.empty(world * n, dtype=pack.dtype, device=pack.device)
                gather_state["e2e_n"] = n
            dist.all_gather_into_tensor(gather_state["e2e_buf"], pack)
    list(pred.predict_batches([waves] * 3, device_hook=hook))
    h0, d0 = eng.h2d_bytes, eng.d2h_bytes
    barrier()
    t0 = time.perf_counter()
    for res in pred.predict_batches((waves for _ in range(args.steps)), device_hook=hook):
        pass
    torch.cuda.synchronize(dev)
    e2e_s = (time.perf_counter() - t0) / args.steps
    t = torch.tensor([e2e_s, sync_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s, sync_s = float(t[0].item()), float(t[1].item())
    h2d = (eng.h2d_bytes - h0) // args.steps
    d2h = (eng.d2h_bytes - d0) // args.steps

    # ---- roofline of the dominant kernel (the FFN GEMMs), CUDA events around each launch -----------------
    roof = None
    shares = None
    if rank == 0:
        eng.profile(True)
        for _ in range(2):
            flush.zero_()
            device_step(eager=True, gather=False)      # rank-0-only leg: no collective here
        torch.cuda.synchronize(dev)
        summ = eng.profile_summary()
        eng.profile(False)
        pk = peaks()
        M = BATCH_PER_GPU * T
        n_ffn = summ["ffn_w1"][0] + summ["ffn_w2"][0]
        ffn_ms_eager = (summ["ffn_w1"][1] + summ["ffn_w2"][1]) / n_ffn      # event pairs around single eager launches (incl. launch latency)
        # the FFN launches back to back from a CUDA graph (as they run inside the timed step), events around the replay
        ffn_ms = ffn_ms_eager
        if eng.gemm_path == "tc" and resident is not None:
            ffn_ms = eng.time_ffn_gemms(resident.g["ws"], int(resident.g["ws"]["x"].shape[0]))   # the step's own row count (incl. frame padding)
        flops = 2.0 * M * 256 * 2048                 # per launch (w_1 and w_2 have the same FLOPs)
        achieved = flops / (ffn_ms * 1e-3) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("ffn_gemm_dram_bytes_per_launch")
            except Exception:
                traffic = None
        kname = ("tc_gemm_kernel (FFN w_1/w_2; tcgen05 kind::f16, FP16x2 split = 3 MMAs per K-step, fp32-grade)"
                 if eng.gemm_path == "tc" else "sgemm_tn_kernel<128,128> (FFN w_1/w_2, fp32 FMA pipe)")
        roof = {"kernel": kname, "bound": "tensor", "achieved": achieved,
                "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_tflops_sustained"],
                "traffic": traffic, "peak_source": pk["source"] + " bf16 sustained", "launch_ms": ffn_ms,
                "launch_ms_eager_event_pairs": ffn_ms_eager,
                "timing": "mean over 24 FFN GEMM launches (w_1, w_2 of block 0 alternating) replayed back to back from a CUDA "
                          "graph, CUDA events around the replay, best of 5; launch_ms_eager_event_pairs = event pairs around "
                          "single eager launches of all 48 FFN GEMMs of a step (includes per-launch latency)",
                "flops_per_launch": flops}
        tot = sum(v[1] for v in summ.values())
        shares = {k: round(v[1] / tot, 4) for k, v in sorted(summ.items(), key=lambda kv: -kv[1][1])}

    # ---- CPU baseline (oracle port) on the host cores: rank 0, N=1 only --------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import conformer as oc
        sd = synth.to_torch(sdn)
        vocab = synth.vocabulary(VOCAB)
        n = args.cpu_baseline_utts
        cores = best_cpu_threads(sd, oc.ConformerConfig(), waves[:1], vocab)
        t0 = time.perf_counter()
        ref = cpu_reference_pass(sd, oc.ConformerConfig(), waves[:n], vocab)
        dt = time.perf_counter() - t0
        res = eng.transcribe(waves[:n])
        same = all(r[2] == tk for r, tk in zip(ref, res.tokens))
        cpu = {"value": n * UTT_SAMPLES / SAMPLE_RATE / dt, "unit": "audio-s/s", "cores": cores, "kind": "port",
               "sample": f"{n} of the 32 utterances (10 s each), B=1 loop fbank->encoder->greedy, torch CPU threads={cores} (best of 4..all)",
               "token_ids_match_gpu": bool(same)}

    if rank == 0:
        line = {"metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 (GEMMs: fp16x2-split operands on tcgen05, fp32 accumulate; fp32-grade results)" if eng.gemm_path == "tc" else "f32",
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "cuda_graph": bool(eng.use_graphs), "global_batch": BATCH_PER_GPU * world, "parallelism": f"dp{world} (utterance shard)",
                           "l2": "flushed between timed steps (256 MiB memset outside the event bracket)",
                           "weights": "synthetic seed 0 (masr_b200.synth)", "wall_ms_per_step_incl_flush": wall * 1e3 / args.steps},
                "e2e": {"value": world * audio_s_rank / e2e_s, "unit": "audio-s/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s * 1e3,
                        "api": "MASRPredictor.predict_batches(iterable of lists of float32 ndarrays) -> lists of {'text','score'}; "
                               "staging + H2D of batch k+1 overlap the GPU pass of batch k",
                        "sync_call": {"value": world * audio_s_rank / sync_s, "ms_per_step": sync_s * 1e3,
                                      "api": "MASRPredictor.predict_batch(list) — one blocking call per batch"}},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "kernel_time_shares": shares,
                "cpu_baseline": cpu}
        if world > 1:
            line["gather_verified"] = gather_verified
            line["config"]["cpu_affinity"] = numa
            line["config"]["collective"] = ("all_gather_into_tensor of the packed int32 outputs, captured in the step's CUDA graph"
                                            if graph_gather else "all_gather_into_tensor of the packed int32 outputs after the graph replay")
            line["strong_scaling"] = strong
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        if graph_gather:
            # CUDA graphs that captured NCCL kernels still reference the communicator; destroy_process_group() then waits
            # forever (seen at N=2, r02).  Everything is measured and printed: leave without tearing NCCL down.
            os._exit(0)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
