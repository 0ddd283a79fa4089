#!/usr/bin/env python
"""bench.py — RTFx of the CrisperWhisper inference-and-alignment path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo (libcrisper.so kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own path: HF pipeline on the host CPU
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs as DIR/<name>.npy

Workload: one GPU = BASELINE.json configs[1] (batch = 8 x 30 s synthetic 16 kHz chunks); several GPUs = configs[3]'s share
(32 chunks per GPU, round-robin, decode batches of 16, transcript all_gather inside the timed region).  CrisperWhisper-
large-v3-shaped random-init weights, greedy decode of a FIXED, STATED number of new tokens (EOS suppressed so both arms do
identical work — RTFx is proportional to 1/T in the decode), 20 alignment heads, median 7, DTW.  `stages` carries configs[2]
(10 min clip), configs[4] (1024-utterance DTW, sharded over the ranks), the whole-encoder tensor roofline and the other
decode batch.
A step = one pass of the whole hot path (log-mel -> encoder -> cross-K/V -> greedy decode -> normalise/median/DTW) over
one batch.  `value` = device-timed throughput with the waveforms already resident in HBM; `e2e` = the same metric
through the public `pipeline(...)` call with HOST numpy waveforms in and the {"text","chunks"} dict out.
Timing: CUDA events on the engine stream, barrier + synchronize on both sides, max over ranks; W >= 3 warm-up steps; every
step's working set (3.1 GB weights + 2 GB cross-K/V + activations) exceeds the 126 MB L2, so no explicit L2 flush is needed.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RTFx (audio-s/s) on 30s chunks, log-mel + Whisper large-v3 greedy decode + DTW word alignment"
UNIT = "audio-s/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]), tf_sust=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    src="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def big_tokenizer(cfg):
    """A synthetic WhisperTokenizer with the large-v3 id layout (51866 ids; real tokenizer files are not available
    offline): byte symbols + made-up text tokens up to 50256, Whisper specials from 50257, timestamps from 50365."""
    from tokenizers import AddedToken
    from tokenizers.pre_tokenizers import ByteLevel
    from transformers import WhisperTokenizer
    from transformers.models.whisper.tokenization_whisper import LANGUAGES
    alphabet = sorted(ByteLevel.alphabet())
    vocab = {ch: i for i, ch in enumerate(alphabet)}
    letters = "abcdefghijklmnopqrstuvwxyz"
    i = 0
    while len(vocab) < cfg["eos_id"]:  # made-up word pieces; every third one starts a new word ("Ġ" = space)
        piece = ("Ġ" if i % 3 == 0 else "") + "".join(letters[(i // 26 ** k) % 26] for k in range(4))
        if piece not in vocab:
            vocab[piece] = len(vocab)
        i += 1
    specials = ["<|endoftext|>", "<|startoftranscript|>"] + [f"<|{l}|>" for l in LANGUAGES] + \
               ["<|translate|>", "<|transcribe|>", "<|startoflm|>", "<|startofprev|>", "<|nospeech|>", "<|notimestamps|>"]
    for s in specials:
        vocab[s] = len(vocab)
    tok = WhisperTokenizer(vocab=vocab, merges=[], language="en", task="transcribe", additional_special_tokens=specials[1:])
    tok.add_tokens([AddedToken("<|%.2f|>" % (k * 0.02), special=False, normalized=False) for k in range(1501)])
    tok.pad_token = "<|endoftext|>"
    assert len(tok) == cfg["vocab"], (len(tok), cfg["vocab"])
    return tok


def synth_wave(seed: int, n: int = 480000) -> np.ndarray:
    return (np.random.default_rng(seed).standard_normal(n) * 0.1).astype(np.float32)


def write_outputs(out_dir: str, arrays: dict, limit: int = 64_000_000) -> None:
    """Save each [chunks, ...] array as out_dir/<name>.npy in float32 (token ids and frame indices are exact there).
    Past `limit` bytes in all, every array keeps the same seeded sample of chunks, whose indices go to chunk_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.cpu().numpy().astype(np.float32) for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(a[0].nbytes for a in host.values()) + 4
    keep = min(n, (limit - 4096) // row_bytes)
    if keep < n:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        host = {k: a[idx] for k, a in host.items()}
        host["chunk_index"] = idx.astype(np.float32)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's own implementation of the path: HF transformers pipeline on the host CPU (REF/transcribe.py:8-34
    with device='cpu', fp32) + REF-equivalent pause adjustment.  Bounded sample per step (stated in the line)."""
    if rank != 0:
        return
    import torch
    from oracle import hf_harness as H
    from oracle import postprocess as PP
    # PyTorch's CPU kernels stop scaling (and then regress badly) beyond a few dozen threads on these small per-token
    # operators: 805 s for one 24-token chunk with 128 threads vs tens of seconds with 16 — use at most 16 and say so
    cores = min(os.cpu_count() or 1, args.ref_threads)
    torch.set_num_threads(cores)
    T = min(args.new_tokens, args.ref_tokens)
    t0 = time.time()
    hf_cfg = H.large_v3_hf_config()
    ids = dict(eos=50257, sot=50258, en=50259, translate=50359, transcribe=50360, no_timestamps=50364)
    heads = [[l, (7 * l) % 20] for l in range(12, 32)]
    # fixed-length single-pass decode on both arms: EOS and every timestamp token but <|0.00|> are suppressed, so the
    # sequence is <|0.00|> + T-1 text tokens and Whisper's seek loop finishes after one encoder/decoder pass
    m = H.build_model(hf_cfg, seed=0, alignment_heads=heads, ids=ids, bf16_round=False, fast_init=True,
                      suppress_tokens=[50257] + list(range(50366, 51866)))
    from crisperwhisper_b200 import weights as Wt
    tok = big_tokenizer(Wt.large_v3_config())
    pipe = H.build_pipeline(m, tok, batch_size=1)
    build_s = time.time() - t0
    wave = synth_wave(0)
    gk = {"max_new_tokens": T}
    import warnings
    times = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for i in range(args.ref_warmup + args.steps):
            t1 = time.perf_counter()
            out = pipe(wave.copy(), generate_kwargs=gk)
            PP.adjust_pauses(out)
            dt = time.perf_counter() - t1
            if i >= args.ref_warmup:
                times.append(dt)
    ms = 1000.0 * float(np.mean(times))
    val = 30.0 / (ms / 1000.0)
    sample = f"1 chunk x 30 s, {T} new tokens (EOS + timestamps suppressed -> one generate pass), HF pipeline fp32 on {cores} host threads"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.ref_warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "reference CPU path, bounded sample of cfg2", "new_tokens": T, "batch_per_step": 1, "host_threads": cores,
                       "model": "whisper-large-v3 shape, random init", "build_s": round(build_s, 1)},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def traffic_from_profile():
    """DRAM bytes of one launch of the dominant kernel, read from the committed ncu summary of this round (profiles/)."""
    p = os.path.join(ROOT, "profiles", "r02_decode_stream_ncu.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    return d, os.path.relpath(p, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="crisper", choices=["crisper", "reference"])
    ap.add_argument("--chunks-per-gpu", dest="chunks", type=int, default=0,
                    help="30 s chunks per GPU per step; default 8 on one GPU (BASELINE cfg 2), 32 on several (cfg 4: 256 chunks over 8 GPUs)")
    ap.add_argument("--batch", type=int, default=0, help="decode batch (chunks per cw_decode_greedy call); default 8 (cfg 2) / 16 (cfg 4 share)")
    ap.add_argument("--new-tokens", dest="new_tokens", type=int, default=445, help="decoded tokens per chunk (445 = n_text_ctx - prompt)")
    ap.add_argument("--ref-tokens", dest="ref_tokens", type=int, default=32, help="decode length of the bounded CPU sample")
    ap.add_argument("--ref-threads", dest="ref_threads", type=int, default=16, help="host threads for the reference arm")
    ap.add_argument("--ref-warmup", dest="ref_warmup", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-stage / per-config measurements")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write the last step's tokens and DTW jump indices of every chunk to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "crisper":
        ap.error("--dump-outputs applies to --impl crisper")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CrisperWhisper hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # the library __graft_entry__.build() left in the tree; the bench never compiles, so the tree may be read-only
    from crisperwhisper_b200 import _lib as L
    from crisperwhisper_b200 import distributed as D
    from crisperwhisper_b200 import weights as Wt
    from crisperwhisper_b200 import adjust_pauses_for_hf_pipeline_output
    from crisperwhisper_b200.engine import Engine
    from crisperwhisper_b200.asr_pipeline import mel_filters_slaney, pipeline

    eng = Engine(local_rank)
    dev = eng.device
    cfg = Wt.large_v3_config(n_align_heads=20, median_filter_width=7)
    cfg["suppress_tokens"] = [50257] + list(range(50366, 51866))  # same fixed-length, single-pass decode as the reference arm
    pw = Wt.synthetic_weights(cfg, dev, seed=0) if rank == 0 else None
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    pw = D.broadcast_weights(pw, cfg, dev)
    torch.cuda.synchronize()
    bcast_ms = (time.perf_counter() - t1) * 1000.0
    eng.load_weights(pw)
    T = args.new_tokens
    NC = args.chunks or (8 if world == 1 else 32)          # chunks per GPU per step
    Bd = args.batch or (8 if NC <= 8 else 16)              # decode batch
    n_prompt = 3
    filt = torch.from_numpy(mel_filters_slaney(128)).to(dev)
    flags = L.CW_DEC_SUPPRESS_EOS
    peaks = measured_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def run_chunks(wave_dev, bd, tnew, gather):
        """stages 1-3 over the resident waveforms [n, 480000] in decode batches of bd; with `gather`, the transcripts'
        device records are all-gathered at the end (cfg 4's end collective) on the engine stream."""
        outs = []
        for b0 in range(0, wave_dev.shape[0], bd):
            w = wave_dev[b0:b0 + bd]
            nb = w.shape[0]
            _, tm, _ = eng.logmel(w, filt, None, want_f32=False, want_tm=True)
            xkv, _ = eng.encode(tm)
            prompt = torch.tensor([[50258, 50259, 50360]] * nb, dtype=torch.int32, device=dev)
            out = eng.decode(xkv, prompt, tnew, flags=flags)
            jump = eng.align(out["align"], torch.full((nb,), tnew - 1, dtype=torch.int32, device=dev),
                             torch.full((nb,), 1500, dtype=torch.int32, device=dev), 7)
            outs.append((out["tokens"], jump))
        if gather and world > 1:
            with torch.cuda.stream(eng.stream):
                toks = torch.cat([o[0] for o in outs]).contiguous()
                jmp = torch.cat([o[1] for o in outs]).contiguous()
                gt = [torch.empty_like(toks) for _ in range(world)]
                gj = [torch.empty_like(jmp) for _ in range(world)]
                dist.all_gather(gt, toks)
                dist.all_gather(gj, jmp)
        return outs

    def time_local(fn, steps, warm):
        """CUDA-event timing on this rank only (no collective: safe in the rank-0-only part of the script)."""
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(eng.stream)
        for _ in range(steps):
            fn()
        e1.record(eng.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    # ---- headline: device-timed step -----------------------------------------------------------------------------------
    waves_host = [synth_wave(i * world + rank) for i in range(NC)]            # chunk i -> rank i mod W (cfg 4 layout)
    wave_dev = torch.from_numpy(np.stack(waves_host)).to(dev)
    for _ in range(max(args.warmup, 3)):
        run_chunks(wave_dev, Bd, T, gather=True)
    barrier()
    launches0 = eng.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(eng.stream)
    for _ in range(args.steps):
        outs = run_chunks(wave_dev, Bd, T, gather=True)
    ev1.record(eng.stream)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:
        dumped = {"tokens": torch.cat([o[0] for o in outs]), "jump_indices": torch.cat([o[1] for o in outs])}
        if world > 1:   # every rank's chunks in global order: local chunk i of rank r is chunk i * world + r
            for k, t in dumped.items():
                parts = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(parts, t)
                dumped[k] = torch.stack(parts, 1).flatten(0, 1)
        if rank == 0:
            write_outputs(args.dump_outputs, dumped)
    gpu_launches = eng.launch_count() - launches0
    ms_per_step = max_over_ranks(ev0.elapsed_time(ev1) / args.steps)
    audio_s = 30.0 * NC * world
    value = audio_s / (ms_per_step / 1000.0)

    # ---- e2e through the public API: host numpy in, {"text","chunks"} out on rank 0 -----------------------------------------
    tok = big_tokenizer(cfg)
    pipe = pipeline("automatic-speech-recognition", model=eng, tokenizer=tok, feature_extractor=None, chunk_length_s=30,
                    batch_size=Bd, return_timestamps="word")
    gk = {"max_new_tokens": T}

    def e2e_step():
        if world == 1:
            res = pipe(waves_host, generate_kwargs=gk)
            return [adjust_pauses_for_hf_pipeline_output(r) for r in res], pipe.last_stats
        # cfg 4: every rank runs stages 1-3 on its round-robin share, the per-chunk records are all-gathered, rank 0 turns
        # all of them into words (tokenizer-level _decode_asr restatement) and adjusts the pauses
        mo = pipe.forward(waves_host, generate_kwargs=gk)
        st = dict(pipe.last_stats)
        local = [(o[0]["tokens"][0], o[0]["token_timestamps"][0]) for o in mo]
        full = D.gather_results(local, NC * world, dev)
        st["d2h_bytes"] = st.get("d2h_bytes", 0) + sum(a.nbytes + b.nbytes for a, b in full)
        res = None
        if rank == 0:
            res = []
            for tk, ts in full:
                r = pipe.postprocess([{"tokens": tk[None, :], "token_timestamps": ts[None, :], "is_last": True, "stride": (480000, 0, 0)}])
                res.append(adjust_pauses_for_hf_pipeline_output(r))
        return res, st

    for _ in range(2):
        e2e_step()
    barrier()
    e2e_times = []
    for _ in range(max(2, min(args.steps, 5))):
        barrier()
        tt = time.perf_counter()
        res, st = e2e_step()
        torch.cuda.synchronize()
        e2e_times.append(max_over_ranks(time.perf_counter() - tt))
    e2e_s = float(np.median(e2e_times))
    e2e_val = audio_s / e2e_s

    # ---- cfg 5 on every rank: 1024 utterances x 20 heads x 448 x 1500, sharded N ways ------------------------------------------
    stages = {}
    if not args.no_extras:
        n_utt = 1024 // world
        sub = 128
        al_buf = torch.empty(sub, 20, 448, 1500, dtype=torch.float32, device=dev)
        Tl = torch.full((sub,), 448, dtype=torch.int32, device=dev)
        Fl = torch.full((sub,), 1500, dtype=torch.int32, device=dev)
        tt = torch.arange(448, device=dev, dtype=torch.float32)[None, None, :, None]
        ff = torch.arange(1500, device=dev, dtype=torch.float32)[None, None, None, :]
        peak_term = 6.0 * torch.exp(-(((ff - tt * 1500.0 / 448.0) / 20.0) ** 2))
        gen = torch.Generator(device=dev)
        tot_ms = 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(0, n_utt, sub):
            gen.manual_seed(1000 * rank + i)
            for j in range(0, sub, 8):   # softmax_F(3 z + 6 exp(-((f - t F/T)/20)^2)), generated on the device (SURVEY 8d cfg 5)
                z = torch.randn(8, 20, 448, 1500, generator=gen, device=dev)
                al_buf[j:j + 8] = torch.softmax(3.0 * z + peak_term, -1)
            if i == 0:
                eng.align(al_buf, Tl, Fl, 7)   # warm-up
            torch.cuda.synchronize(dev)        # the generator above ran on torch's stream: keep it out of the timed region
            e0.record(eng.stream)
            eng.align(al_buf, Tl, Fl, 7)
            e1.record(eng.stream)
            eng.sync()
            tot_ms += e0.elapsed_time(e1)
        del al_buf, z
        dtw_ms = max_over_ranks(tot_ms)
        dtw_bytes = 1024 * (20 * 448 * 1500 * 4 + 448 * 4)
        stages["dtw_cfg5"] = {"workload": f"cfg5: 1024 utterances x 20 heads x 448 x 1500 f32, {n_utt} per GPU on {world} GPU(s), in resident sub-batches of {sub}",
                              "ms_max_over_ranks": round(dtw_ms, 3), "achieved_GBs_whole_job": round(dtw_bytes / (dtw_ms * 1e-3) / 1e9, 1),
                              "achieved_GBs_per_gpu": round(dtw_bytes / world / (dtw_ms * 1e-3) / 1e9, 1), "peak_GBs_per_gpu": peaks["hbm"],
                              "frac": round(dtw_bytes / world / (dtw_ms * 1e-3) / 1e9 / peaks["hbm"], 4), "bound": "hbm",
                              "kernels": "align_reduce_kernel + dtw_kernel"}

    # last collective of the run: everything below is rank-0-only and must not touch the process group
    if world > 1:
        dist.barrier()
    if rank != 0:
        dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (rank 0), measured live with CUDA events --------------------------------------------------
    # decode_stream_kernel: one cooperative launch = up to 16 decode steps of the whole decode batch; a decode call of T new
    # tokens is ceil((T + n_prompt - 1) / 16) launches, timed back to back on the engine stream.
    def decode_roofline(bd):
        wv = wave_dev[:bd] if wave_dev.shape[0] >= bd else torch.from_numpy(np.stack([synth_wave(900 + i) for i in range(bd)])).to(dev)
        _, tm, _ = eng.logmel(wv, filt, None, want_f32=False, want_tm=True)
        xkv, _ = eng.encode(tm)
        prompt = torch.tensor([[50258, 50259, 50360]] * bd, dtype=torch.int32, device=dev)
        eng.decode(xkv, prompt, T, flags=flags)
        eng.sync()
        n_steps = T + n_prompt - 1
        n_launch = (n_steps + 15) // 16
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dec_ms = []
        for _ in range(3):
            d0.record(eng.stream)
            eng.decode(xkv, prompt, T, flags=flags)
            d1.record(eng.stream)
            eng.sync()
            dec_ms.append(d0.elapsed_time(d1))
        call_ms = float(np.median(dec_ms))
        d, H, F, Ld, ffn, Vp = cfg["d_model"], cfg["n_heads"], 1500, cfg["dec_layers"], cfg["ffn_dim"], cfg["vocab_padded"]
        w_bytes = Ld * (3 * d * d + 3 * d * d + 2 * d * ffn) * 2 + Vp * d * 2       # qkv, o, q_c, o_c, fc1, fc2 + tied proj_out
        xkv_bytes = Ld * bd * H * F * 2 * 64 * 2                                     # cross K and V of every sample
        self_bytes = Ld * bd * 2 * d * 2 * (n_prompt + T) // 2                       # self KV cache, mean length
        align_bytes = bd * 20 * F * 4                                                # alignment-head rows written
        step_bytes = w_bytes + xkv_bytes + self_bytes + align_bytes
        achieved = step_bytes * n_steps / (call_ms * 1e-3) / 1e9
        return dict(batch=bd, ms_per_decode_step=round(call_ms / n_steps, 4), avg_launch_ms=round(call_ms / n_launch, 3),
                    launches_timed=3 * n_launch, steps_per_launch=16, algorithmic_bytes_per_step=int(step_bytes),
                    achieved=round(achieved, 1), frac=round(achieved / peaks["hbm"], 4), call_ms=call_ms,
                    bytes_breakdown_GB={"decoder_weights": round(w_bytes / 1e9, 3), "cross_kv": round(xkv_bytes / 1e9, 3),
                                        "self_kv_mean": round(self_bytes / 1e9, 3), "alignment_rows": round(align_bytes / 1e9, 4)})

    r = decode_roofline(Bd)
    prof, prof_path = traffic_from_profile()
    traffic = None
    if prof and prof.get("dram_bytes_per_launch") and prof.get("steps_in_launch"):
        traffic = int(prof["dram_bytes_per_launch"] / prof["steps_in_launch"] * 16)
    roofline = {"bound": "hbm", "kernel": "decode_stream_kernel (one cooperative launch = 16 decode steps of the whole decode batch)",
                "achieved": r["achieved"], "peak": peaks["hbm"], "unit": "GB/s", "frac": r["frac"],
                "traffic": traffic,
                "traffic_source": (f"{prof_path}: ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one launch "
                                   f"({prof.get('steps_in_launch')} steps, commit {prof.get('commit')}), scaled to 16 steps") if prof else None,
                "peak_source": peaks["src"] + " (of measured, sustained-copy figure)",
                "algorithmic_bytes_per_launch": int(r["algorithmic_bytes_per_step"] * 16), "avg_launch_ms": r["avg_launch_ms"],
                "ms_per_decode_step": r["ms_per_decode_step"], "launches_timed": r["launches_timed"],
                "bytes_breakdown_GB_per_step": r["bytes_breakdown_GB"], "decode_batch": Bd,
                "share_of_step": round(r["call_ms"] * ((NC + Bd - 1) // Bd) / ms_per_step, 3)}

    alt = None
    if not args.no_extras:
        # ---- other decode batches / lengths, whole-encoder tensor roofline, cfg 3, cfg 4 share ---------------------------------------
        other = 16 if Bd == 8 else 8
        ro = decode_roofline(other)
        stages["decode_other_batch"] = {k: ro[k] for k in ("batch", "ms_per_decode_step", "achieved", "frac")}
        if T != 128:
            w8 = wave_dev[:min(8, NC)]
            t128 = time_local(lambda: run_chunks(w8, min(8, NC), 128, gather=False), 2, 1)
            alt = {"new_tokens": 128, "ms_per_step": round(t128, 2), "value": round(30.0 * w8.shape[0] / (t128 / 1000.0), 1),
                   "note": "8 chunks with 128 new tokens per chunk (typical for 30 s of speech), one GPU; not the headline"}
        # whole encoder + cross-K/V (conv as GEMM, 32 layers, attention, final LN, K/V projection): 2588.4 GFLOP per chunk
        _, tm8, _ = eng.logmel(wave_dev[:min(8, NC)], filt, None, want_f32=False, want_tm=True)
        nb8 = tm8.shape[0]
        enc_ms = time_local(lambda: eng.encode(tm8), 5, 2)
        enc_tf = nb8 * 2588.4e9 / (enc_ms * 1e-3) / 1e12
        stages["encoder_whole"] = {"batch": nb8, "ms": round(enc_ms, 3), "achieved_TFLOPs": round(enc_tf, 1), "GFLOP_per_chunk": 2588.4,
                                   "peak_TFLOPs_sustained": peaks["tf_sust"], "frac_of_sustained": round(enc_tf / peaks["tf_sust"], 4),
                                   "peak_TFLOPs_burst": peaks["tf_burst"], "frac_of_burst": round(enc_tf / peaks["tf_burst"], 4), "bound": "tensor"}
        M = nb8 * 1500
        A = (torch.randn(M, 1280, device=dev) * 0.5).to(torch.bfloat16)
        W = (torch.randn(5120, 1280, device=dev) * 0.5).to(torch.bfloat16)
        gms = time_local(lambda: eng.gemm(A, W), 20, 3)
        tf = 2.0 * M * 5120 * 1280 / (gms * 1e-3) / 1e12
        stages["encoder_gemm"] = {"shape": [M, 5120, 1280], "ms": round(gms, 4), "achieved_TFLOPs": round(tf, 1),
                                  "peak_TFLOPs": peaks["tf_burst"], "frac": round(tf / peaks["tf_burst"], 4), "bound": "tensor"}
        del A, W
        if world == 1:
            # cfg 3: 10-minute clip -> 30 chunks (29 x 30 s + 20 s, 5 s strides), batch 16, through the public pipeline incl. the
            # stride merge and the pause adjustment; host waveform in, dict out
            rng = np.random.default_rng(77)
            long_wave = (rng.standard_normal(9600000) * 0.1).astype(np.float32)
            pipe16 = pipeline("automatic-speech-recognition", model=eng, tokenizer=tok, feature_extractor=None, chunk_length_s=30,
                              batch_size=16, return_timestamps="word")
            adjust_pauses_for_hf_pipeline_output(pipe16(long_wave, generate_kwargs=gk))
            lt = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                o3 = adjust_pauses_for_hf_pipeline_output(pipe16(long_wave, generate_kwargs=gk))
                torch.cuda.synchronize()
                lt.append(time.perf_counter() - t0)
            stages["longform_cfg3"] = {"workload": f"cfg3: 10 min clip -> {pipe16.last_stats['chunks']} chunks (30 s / 5 s stride), batch 16, {T} new tokens per chunk, "
                                                   "pipeline(...) + stride merge + adjust_pauses, host in / dict out",
                                       "seconds": round(float(np.median(lt)), 3), "value": round(600.0 / float(np.median(lt)), 1), "unit": UNIT,
                                       "words": len(o3["chunks"])}
            # cfg 4's per-GPU share on this one GPU (32 chunks, decode batch 16) so that the N-GPU lines can be compared at equal work
            w32 = torch.from_numpy(np.stack([synth_wave(500 + i) for i in range(32)])).to(dev)
            t32 = time_local(lambda: run_chunks(w32, 16, T, gather=False), 2, 1)
            stages["cfg4_share_one_gpu"] = {"workload": f"32 chunks x 30 s per GPU (cfg 4: 256 over 8), decode batch 16, {T} new tokens, device-timed",
                                            "ms_per_step": round(t32, 1), "value": round(960.0 / (t32 / 1000.0), 1), "unit": UNIT}
            del w32

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:   # the CPU baseline is timed on rank 0 at N = 1 only
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--new-tokens",
                                  str(T), "--ref-tokens", str(args.ref_tokens), "--ref-threads", str(args.ref_threads)],
                                 capture_output=True, text=True, timeout=900,
                                 env={**os.environ, "RANK": "0", "WORLD_SIZE": "1", "CUDA_VISIBLE_DEVICES": ""})
            ref_line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
            cpu_baseline = ref_line["cpu_baseline"]
            cpu_baseline["kind"] = "reference"
        except Exception as e:  # pragma: no cover
            cpu_baseline = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e}"}

    wl = (f"cfg2: batch={NC} x 30 s synthetic 16 kHz chunks on one GPU" if world == 1 else
          f"cfg4 share: {NC} x 30 s chunks per GPU ({NC * world} chunks round-robin over {world} GPUs), decode batches of {Bd}, transcript "
          "all_gather inside the timed region (e2e: + word decoding of all chunks on rank 0)")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": wl + f", CrisperWhisper large-v3 shape (random init), greedy decode {T} new tokens (EOS suppressed) + "
                                    "20-head median-7 DTW alignment",
                   "new_tokens": T, "chunks_per_gpu": NC, "decode_batch": Bd, "global_chunks": NC * world,
                   "parallelism": f"dp{world} (chunk i -> rank i mod {world})",
                   "l2": "working set per step (3.1 GB weights + 1.7 GB fragment-major copies + 2-4 GB cross-K/V) >> 126 MB L2; no explicit flush",
                   "weights_broadcast_ms": round(bcast_ms, 2),
                   "note": "one GPU measures cfg 2 (8 chunks); several GPUs measure cfg 4's share (32 chunks per GPU); "
                           "stages.cfg4_share_one_gpu gives the one-GPU number at the multi-GPU per-GPU work"},
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(st.get("h2d_bytes", 0)),
                "d2h_bytes_per_step": int(st.get("d2h_bytes", 0)),
                "api": "crisperwhisper_b200.pipeline(...)(list of np.ndarray) + adjust_pauses" if world == 1 else
                       "pipeline.forward(host chunks) per rank + distributed.gather_results + pipeline.postprocess + adjust_pauses on rank 0",
                "ms_per_step": round(e2e_s * 1000.0, 2)},
        "gpu_launches": int(gpu_launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline, "stages": stages,
        "alt_decode_length": alt,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
