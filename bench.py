#!/usr/bin/env python
"""bench.py - S2ST utterances/sec for seamlessM4T_v2_large + vocoder_v2 on B200 (BASELINE.json metric).

A "step" is one pass of the whole hot path (fbank -> Conformer encoder -> beam-search text decoder -> NAR T2U ->
Code-HiFiGAN) over one batch of 32 x 10 s synthetic 16 kHz utterances per GPU through `Translator.predict`, with
random-init weights of the named architecture (no checkpoints are reachable offline).

  value : utt/s with the input waveforms already resident in HBM when the timed region starts
  e2e   : the same through the public API with HOST (pinned) waveforms: every step copies its inputs host -> device and
          its waveforms / units device -> host inside the timed region; the copies (and, for N>1, the NCCL scatter of
          inputs from rank 0 / gather of waveforms to rank 0) run on side streams under the neighbouring steps' compute
          (seamless_communication_b200/parallel.py: OverlappedExchange)
  roofline     : the time-dominant stage - one beam-search step (HBM bound: decoder + tied-projection weights, K/V) -
                 measured live; `stages` holds every stage against its own bound
  parity       : the GPU path against the fp32 oracle on the first utterance of the batch (the oracle run that also
                 provides cpu_baseline)
  cpu_baseline : the fp32 CPU oracle (a port of the reference path; the reference's fairseq2 stack is not installable
                 offline) on a bounded sample, on this box's host cores; knf (the reference's own C++ fbank) timed apart
  --impl reference : times that CPU path as the reference arm (batch 4, 1 warm-up + K timed runs).
  --config s2tt    : BASELINE configs[1] (8 x 10 s, encoder + text decoder only).
  --config stream  : BASELINE configs[4] (SeamlessStreaming EMMA S2ST, one 30 s synthetic stream in 320 ms segments): compute
                     latency per source segment and the real-time factor.
  --dump-outputs DIR : after the timed steps, writes what the last timed step returned to its caller as DIR/<name>.npy
                     (dump_outputs).  Inputs and weights are seeded, so two builds run with the same arguments can be
                     compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TGT_LANG, LANG_IDX, SPKR_IDX = "spa", 25, 45
SAMPLES, HARD_MAX, BEAM = 160000, int(os.environ.get("SB_BENCH_HARD_MAX", "102")), 5
CONFIGS = {
    "s2st": dict(batch=32, task="s2st", metric="s2st_utterances_per_sec",
                 workload="S2ST seamlessM4T_v2_large + vocoder_v2, batch 32x10s synthetic 16 kHz per GPU, beam 5, "
                          "hard_max_seq_len 102 (L=102 text tokens, U=495 units, 9.9 s out) [BASELINE configs[2]]"),
    "s2tt": dict(batch=8, task="s2tt", metric="s2tt_utterances_per_sec",
                 workload="S2TT seamlessM4T_v2_large, batch 8x10s synthetic 16 kHz per GPU, beam 5, hard_max_seq_len 102 "
                          "(Conformer encoder + text decoder only) [BASELINE configs[1]]"),
}
STREAM_WORKLOAD = ("SeamlessStreaming S2ST (EMMA monotonic text decoder dense_1b + seamlessM4T_v2_large encoder / NAR T2U + "
                   "vocoder_v2), one 30 s synthetic 16 kHz stream fed in 320 ms segments, reference evaluation defaults "
                   "(cli/streaming/evaluate.py:55-66) [BASELINE configs[4]]")
# algorithmic work per 10 s utterance at L=102, U=495 (SURVEY 8d / BASELINE.md 2)
GFLOP_PER_UTT = {"encoder": 618.9, "t2u": 155.0, "vocoder": 165.0}
FBANK_BYTES_PER_UTT = 0.80e6
DUMP_BYTES = 60 << 20  # array data written by --dump-outputs, all files together


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"{s} is not >= 1")
    return v


def dump_outputs(out_dir, texts=None, text_ids=None, units=None, wavs=None):
    """Writes one step's outputs as out_dir/<name>.npy: texts as Unicode code points and token / unit ids as float64
    (exact), waveforms as float32.  Each is a list of 1-D rows, stored padded to a rectangle (-1 for ids, 0 for audio)
    with the row lengths in <name>_lengths.npy.  If the waveforms would take the data past DUMP_BYTES, a fixed seeded
    sample of their time positions is kept, listed in audio_wavs_positions.npy."""
    import numpy as np

    def rect(rows, pad, dtype):
        lens = np.array([len(r) for r in rows], dtype=np.float64)
        a = np.full((len(rows), int(lens.max(initial=0))), pad, dtype=dtype)
        for i, r in enumerate(rows):
            a[i, :len(r)] = r
        return a, lens

    arrays = {}
    if texts is not None:
        arrays["texts"], arrays["texts_lengths"] = rect([[ord(c) for c in t] for t in texts], -1, np.float64)
    if text_ids is not None:
        arrays["text_ids"], arrays["text_ids_lengths"] = rect(text_ids, -1, np.float64)
    if units is not None:
        arrays["units"], arrays["units_lengths"] = rect(units, -1, np.float64)
    if wavs is not None:
        w, lens = rect([x.detach().flatten().float().cpu().numpy() for x in wavs], 0, np.float32)
        room = DUMP_BYTES - sum(a.nbytes for a in arrays.values()) - lens.nbytes
        if w.nbytes > room:
            keep = room // (4 * w.shape[0] + 8)
            pos = np.sort(np.random.default_rng(0).choice(w.shape[1], size=keep, replace=False))
            w, arrays["audio_wavs_positions"] = w[:, pos], pos.astype(np.float64)
        arrays["audio_wavs"], arrays["audio_wavs_lengths"] = w, lens
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(sm)}


def build_models(device):
    from seamless_communication_b200 import config as C, synthetic as S
    from seamless_communication_b200.inference import Translator
    from seamless_communication_b200.models.unity import load_unity_model
    from seamless_communication_b200.models.vocoder import load_vocoder_model

    cfg, vc = C.base_v2(), C.base_vocoder()
    sd = S.make_unity_state_dict(cfg, seed=0, dec_gain=4.0)
    vsd = S.make_vocoder_state_dict(vc, seed=1)
    toks = S.make_tokenizers(cfg)
    model = load_unity_model("seamlessM4T_v2_large", device=device, state_dict=sd, tokenizers=toks)
    voc = load_vocoder_model("vocoder_v2", device=device, state_dict=vsd)
    return Translator(model, voc, device=device)


# ------------------------------------------------------------------------------------------------ CPU reference arm
_ORACLE = {}


def _oracle_models():
    if not _ORACLE:
        from oracle.unity_oracle import UnityOracle, VocoderOracle
        from seamless_communication_b200 import config as C, synthetic as S
        cfg, vc = C.base_v2(), C.base_vocoder()
        toks = S.make_tokenizers(cfg)
        _ORACLE["uo"] = UnityOracle(cfg.to_dict(), S.make_unity_state_dict(cfg, seed=0, dec_gain=4.0), toks)
        _ORACLE["vo"] = VocoderOracle(vc.to_dict(), S.make_vocoder_state_dict(vc, seed=1))
        _ORACLE["toks"] = toks
    return _ORACLE["uo"], _ORACLE["vo"], _ORACLE["toks"]


def pick_cpu_threads():
    """BASELINE.md 3: "all cores" is not the fastest setting for this path - the host-driven beam search multiplies 5-row
    matrices and torch's CPU GEMMs slow down with too many threads on such shapes.  Probe {16, 32, 64, 128, all} on a
    short search and keep the fastest; the count used is reported as `cores`."""
    from oracle.unity_oracle import fbank
    from seamless_communication_b200 import synthetic as S
    uo, _, toks = _oracle_models()
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, 128, cores) if c <= cores})
    w = S.make_waveforms(1, 32000, seed=1)
    best, best_t, probe = cands[0], float("inf"), {}
    with torch.inference_mode():
        for c in cands:
            torch.set_num_threads(c)
            fb = fbank(w[0])[None]
            enc, _ = uo.encode_speech(fb, None)
            t0 = time.time()
            uo.beam_search(enc, None, [3, toks[0].lang_index(TGT_LANG)], hard_max=5)
            dt = time.time() - t0
            probe[c] = round(dt, 3)
            if dt < best_t:
                best, best_t = c, dt
    return best, probe


def cpu_oracle_run(n_utts, threads, task="s2st", trace=None):
    """The reference CPU path (oracle port) on n_utts utterances of the bench workload.
    Returns (seconds, utt/s, outputs, per-stage seconds)."""
    from oracle.unity_oracle import s2st
    from seamless_communication_b200 import synthetic as S

    uo, vo, _ = _oracle_models()
    torch.set_num_threads(threads)
    waves = S.make_waveforms(n_utts, SAMPLES, seed=1234)
    timers = {}
    with torch.inference_mode():
        t0 = time.time()
        if task == "s2st":
            out = s2st(uo, vo, waves, TGT_LANG, LANG_IDX, SPKR_IDX, hard_max=HARD_MAX, timers=timers, trace=trace)
        else:
            from oracle.unity_oracle import fbank
            t1 = time.time()
            fb = torch.stack([fbank(w) for w in waves])
            timers["fbank"] = time.time() - t1
            out = uo.generate(fb, None, TGT_LANG, hard_max=HARD_MAX, output_units=False, timers=timers, trace=trace)
        dt = time.time() - t0
    return dt, n_utts / dt, out, {k: round(v, 3) for k, v in timers.items()}


def knf_fbank_seconds(n_utts=4):
    """The reference's own C++ fbank (kaldi-native-fbank, compiled in place into oracle/_ref/libknf_ref.so), single thread,
    one utterance at a time as fairseq2n calls it (BASELINE.md 3.2).  Seconds per 10 s utterance, or None."""
    so = os.path.join(ROOT, "oracle", "_ref", "libknf_ref.so")
    if not os.path.exists(so):
        return None
    from seamless_communication_b200 import synthetic as S
    lib = ctypes.CDLL(so)
    lib.knf_fbank.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p]
    waves = S.make_waveforms(n_utts, SAMPLES, seed=1234).contiguous()
    out = torch.empty(1000, 80)
    lib.knf_fbank(waves[0].data_ptr(), SAMPLES, 32768.0, out.data_ptr())  # warm-up
    t0 = time.time()
    for i in range(n_utts):
        lib.knf_fbank(waves[i].data_ptr(), SAMPLES, 32768.0, out.data_ptr())
    return (time.time() - t0) / n_utts


def cpu_baseline_block(task, batch, timed_runs, warmup=True, trace=None):
    threads, probe = pick_cpu_threads()
    if warmup:
        cpu_oracle_run(1, threads, task)  # first-touch of 9 GB of fp32 weights, thread pool spin-up
    runs, out, stages = [], None, None
    for _ in range(timed_runs):
        dt, _, out, stages = cpu_oracle_run(batch, threads, task, trace=trace)
        runs.append(dt)
    dt = statistics.mean(runs)
    knf = knf_fbank_seconds()
    block = {"value": batch / dt, "unit": "utt/s", "cores": threads, "kind": "port", "host_cores": os.cpu_count(),
             "rtf": dt / (10.0 * batch), "batch": batch, "seconds_per_run": [round(x, 2) for x in runs],
             "stages_s": stages, "thread_probe_s": probe,
             "knf_fbank_s_per_utt": None if knf is None else round(knf, 4),
             "sample": f"{batch} x 10 s utterances ({task}, full model, beam 5, L=102) through the fp32 CPU oracle, "
                       f"{'1 warm-up + ' if warmup else ''}{timed_runs} timed run(s); thread count = fastest of the probe; "
                       "batch 32 of BASELINE.md 3.5 is not run inside the default time box (decoding is per sentence on the "
                       "CPU path, so utt/s at batch 32 equals batch 4 to within the encoder's batching gain)"}
    return block, out


def workload_config(cfg, batch, world):
    """`config` of the bench line: the workload only, identical in both arms (how this arm runs it is under `pipeline`)."""
    return {"workload": cfg["workload"], "per_gpu_batch": batch, "global_batch": batch * world, "parallelism": f"dp{world}",
            "l2": "working set (3.5 GB fp16 weights + activations) >> 126 MB L2, no explicit flush",
            "weights": "random-init, seeded", "accumulate": "f32"}


def run_reference(args, rank):
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    block, out = cpu_baseline_block(cfg["task"], 4, args.steps, warmup=args.warmup > 0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, texts=out["texts"], units=out.get("speech_units"), wavs=out.get("wavs"))
    v = block["value"]
    line = {"impl": "reference", "metric": cfg["metric"], "value": v, "unit": "utt/s", "n_gpus": args.gpus,
            "steps": len(block["seconds_per_run"]), "warmup": 1 if args.warmup > 0 else 0,
            "ms_per_step": 1e3 * statistics.mean(block["seconds_per_run"]), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, cfg["batch"], max(1, args.gpus)),
            "sample": "each step = batch 4 of the workload's utterances on the host CPU (BASELINE.md 3 protocol: 1 warm-up, "
                      "--steps timed runs, thread count = fastest of a probe)",
            "cpu_baseline": block,
            "e2e": {"value": v, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm helpers
def stage_times(tr, waves_dev, task):
    """GPU time per stage of one step (CUDA events; not part of the timed region)."""
    eng = tr.model.engine
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    marks = [ev() for _ in range(7)]
    torch.cuda.synchronize()
    marks[0].record()
    src = tr.fbank_batch(waves_dev)
    marks[1].record()
    enc, lens = eng.encode_speech(src["seqs"], None)
    marks[2].record()
    prefix = [eng.cfg.text_eos, eng.text_tokenizer.lang_index(TGT_LANG)]
    hyps = eng.beam_search(enc, None, prefix, beam=BEAM, hard_max=HARD_MAX)
    marks[3].record()
    seqs = [h[0][1] for h in hyps]
    out = {}
    if task == "s2st":
        L = max(len(s) for s in seqs)
        ts = torch.zeros((len(seqs), L), dtype=torch.int64)
        for i, s in enumerate(seqs):
            ts[i, :len(s)] = torch.tensor(s)
        ts = ts[:, :-1].contiguous().to(enc.buf.device)
        dec = eng.harvest_decoder_states([len(s) - 1 for s in seqs])  # same states the search computed (no second pass)
        marks[4].record()
        units, ulens, _ = eng.t2u(dec, ts)
        marks[5].record()
        tr.vocoder(units, TGT_LANG, -1, dur_prediction=False)
        marks[6].record()
        out["units_per_utt"] = int(ulens.max().item())
    torch.cuda.synchronize()
    names = ["fbank", "encoder", "beam_search", "harvest_states", "t2u", "vocoder"][:6 if task == "s2st" else 3]
    out.update({n: marks[i].elapsed_time(marks[i + 1]) for i, n in enumerate(names)})
    out["decode_positions"] = max(len(s) for s in seqs)
    return out


def lanes_search_ms(pool, eng, enc, lanes, reps=2):
    """Time in which `lanes` concurrent beam searches (one per lane, same resident encoder output) complete, ms."""
    prefix = [eng.cfg.text_eos, eng.text_tokenizer.lang_index(TGT_LANG)]
    fn = lambda: eng.beam_search(enc, None, prefix, beam=BEAM, hard_max=HARD_MAX) and None  # noqa: E731
    pool.map(fn, [()] * lanes)
    main = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    futs = [pool.submit(i, fn) for i in range(lanes * reps)]
    for f in futs:
        _, done = f.result()
        main.wait_event(done)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def decode_step_bytes(eng, batch, steps_dec):
    """Algorithmic bytes of ONE beam-search step for the whole batch (SURVEY 8d, DESIGN 3): every decoder weight and the
    tied projection once, the self-attention K/V of all rows at the mean position, the static cross-attention K/V once
    per utterance."""
    R = batch * BEAM
    w_bytes = sum(v.numel() * v.element_size() for k, v in eng.w.items()
                  if k.startswith("text_decoder.") and "encoder_decoder_attn.kv" not in k) + eng.w["text_embed"].numel() * 2
    kv_self = 2 * eng.cfg.dec_layers * R * eng.M * 2 * (steps_dec / 2.0)
    kv_cross = eng.cfg.dec_layers * batch * 63 * 2 * eng.M * 2
    return w_bytes + kv_self + kv_cross, dict(weights=w_bytes, kv_self_mean=kv_self, kv_cross=kv_cross)


def measured_decode_traffic():
    """DRAM bytes of one beam-search step from this round's ncu passes over `bench.py --profile-only` with a 13-step search
    (tools/ncu_summary.py).  Two passes: `--cache-control none` (L2 contents carried from kernel to kernel, as in a real
    step: split-K partials and activations stay in L2) is the figure reported as `traffic`; the default pass flushes the
    caches before every launch, so every intermediate is counted as DRAM traffic (`traffic_cold`)."""
    out = {}
    for key, name in (("warm", "r02warm_decode_step_dram.json"), ("cold", "r02_decode_step_dram.json")):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            out[key] = json.load(open(p))
    return out


def stage_table(stages, batch, pk, eng, task):
    """Every stage against its own bound (tensor stages vs the SUSTAINED bf16 peak: they run inside a long step)."""
    tab = {}
    for name, gf in GFLOP_PER_UTT.items():
        if name in stages:
            tf = gf * batch / stages[name]  # GFLOP / ms = TFLOP/s
            tab[name] = {"ms": stages[name], "bound": "tensor", "algorithmic_gflop": gf * batch, "achieved_tflops": tf,
                         "frac": tf / pk["tf_sustained"]}
    if "fbank" in stages:
        gbs = FBANK_BYTES_PER_UTT * batch / (stages["fbank"] * 1e-3) / 1e9
        tab["fbank"] = {"ms": stages["fbank"], "bound": "hbm", "algorithmic_bytes": FBANK_BYTES_PER_UTT * batch, "achieved_gbs": gbs,
                        "frac": gbs / pk["hbm"]}
    steps_dec = stages["decode_positions"] - 1
    b_step, parts = decode_step_bytes(eng, batch, steps_dec)
    ms_step = stages["beam_search"] / steps_dec
    gbs = b_step / (ms_step * 1e-3) / 1e9
    tab["beam_search"] = {"ms": stages["beam_search"], "bound": "hbm", "steps": steps_dec, "ms_per_step": ms_step,
                          "algorithmic_bytes_per_step": b_step, "bytes_breakdown": parts, "achieved_gbs": gbs, "frac": gbs / pk["hbm"]}
    return tab


def parity_block(tr, ref, waves_dev, task):
    """GPU outputs on utterance 0 of the bench batch against the oracle outputs of the same utterance (bench.py computes
    the oracle run for cpu_baseline anyway).  The strict, staged version is tests/test_gpu_parity.py::test_full_width_*."""
    from seamless_communication_b200.inference import SequenceGeneratorOptions
    eng = tr.model.engine
    M = eng.M
    opts = SequenceGeneratorOptions(beam_size=BEAM, soft_max_seq_len=(1, 200), hard_max_seq_len=HARD_MAX)
    src = tr.fbank_batch(waves_dev[:1])
    texts, speech = tr.predict(src, task, TGT_LANG, text_generation_opts=opts)
    enc = tr.model._last_enc.buf.view(1, -1, M).float().cpu()
    out = {"utterance": "seed 1234 #0", "enc_rel_err": float((enc - ref["enc"][:1]).abs().max() / ref["enc"][:1].abs().max())}
    ids = tr._last_generator.last_text_output.hypotheses[0][0][1]
    ids_o = ref["text_ids"][0]
    out["text_ids_equal"] = bool(ids == ids_o)
    out["text_len"] = len(ids)
    out["text_common_prefix"] = next((i for i, (a, b) in enumerate(zip(ids, ids_o)) if a != b), min(len(ids), len(ids_o)))
    if ids != ids_o:
        # margin audit: the GPU's hypothesis scored by the ORACLE (teacher-forced fp32 pass) against the oracle's own best -
        # a difference within fp16-vs-fp32 logit noise is a near tie of the search, not a defect (oracle/ASSUMPTIONS.md 9)
        uo = _oracle_models()[0]
        with torch.inference_mode():
            t = torch.tensor(ids)[None]
            h = uo.decoder(uo.embed_text(t[:, :-1], 0), ref["enc"][:1], None)
            lp = torch.log_softmax(uo.project(h).float(), -1)[0]
            sc = sum(float(lp[i, t[0, i + 1]]) for i in range(t.shape[1] - 1)) / (t.shape[1] - 1)
        out["oracle_score_of_gpu_hypothesis"] = sc
        out["oracle_best_score"] = float(ref["hyps"][0][0][0])
        out["near_tie"] = bool(abs(sc - out["oracle_best_score"]) < 2e-2)
    if task == "s2st":
        u_ref = ref["speech_units"][0]
        u = speech.units[0]
        out["units_len"] = [len(u), len(u_ref)]
        out["units_differing"] = int(sum(a != b for a, b in zip(u, u_ref)) + abs(len(u) - len(u_ref)))
        if out["units_differing"] and len(u) == len(u_ref) and "logits" in ref:
            # margin audit of the differing units: the oracle's own top-1 / top-2 unit logits at those positions - an fp16
            # argmax can only flip where the fp32 margin is inside the logit noise (4e-2 abs at full width, DESIGN 4)
            try:
                pos = [i for i, (a, b) in enumerate(zip(u, u_ref)) if a != b]
                top2 = ref["logits"][0].float()[pos].topk(2, dim=-1).values
                margins = top2[:, 0] - top2[:, 1]
                out["units_oracle_top2_margin_at_diffs"] = [round(float(m), 4) for m in margins]
                out["units_near_tie"] = bool(float(margins.max()) < 5e-2)
            except Exception as ex:  # the audit must never cost the bench line
                out["units_audit_error"] = repr(ex)
        w, w_ref = speech.audio_wavs[0].float().cpu().flatten(), ref["wavs"][0].flatten()
        n = min(w.numel(), w_ref.numel())
        out["wav_max_abs_err"] = float((w[:n] - w_ref[:n]).abs().max()) if out["units_differing"] == 0 else None
    return out


def run_stream(args, device):
    """BASELINE configs[4]: per-segment compute latency and RTF of the streaming chain (one stream, as the reference runs it)."""
    from seamless_communication_b200 import config as C, synthetic as S
    from seamless_communication_b200.models.monotonic_decoder import load_monotonic_decoder_model
    from seamless_communication_b200.streaming.pipeline import StreamingS2ST

    tr = build_models(device)
    cfg = C.base_v2()
    toks = (tr.model.engine.text_tokenizer, tr.model.engine.char_tokenizer)
    mono = load_monotonic_decoder_model("base_v2", device=device, state_dict=S.make_monotonic_state_dict(cfg, seed=2), tokenizers=toks)
    wave = torch.cat([w for w in S.make_waveforms(3, SAMPLES, seed=4321)])  # 30 s
    results = []
    for rep in range(max(1, args.warmup) + args.steps):
        st = StreamingS2ST(tr.model, mono, tr.vocoder, TGT_LANG)
        torch.cuda.synchronize()
        ids, chunks = st.run(wave)
        results.append(st)
    timed = results[max(1, args.warmup):]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, text_ids=[ids], wavs=[torch.cat([c.flatten() for c in chunks]) if chunks else torch.zeros(0)])
    lat = sorted(x for st in timed for x in st.latencies_ms)
    total_ms = statistics.mean(sum(st.latencies_ms) for st in timed)
    st = timed[-1]
    audio_s = wave.numel() / 16000.0
    q = lambda p: lat[min(len(lat) - 1, int(p * len(lat)))]  # noqa: E731
    line = {"metric": "streaming_s2st_rtf", "value": total_ms * 1e-3 / audio_s, "unit": "s compute / s audio", "n_gpus": 1,
            "steps": len(timed), "warmup": max(1, args.warmup), "ms_per_step": total_ms, "higher_is_better": False, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": STREAM_WORKLOAD, "segments": len(st.latencies_ms), "segment_ms": 320},
            "latency_ms_per_segment": {"mean": statistics.mean(lat), "p50": q(0.5), "p95": q(0.95), "max": lat[-1]},
            "wall_s_per_stream": st.wall_s, "text_tokens": len(st.text_ids),
            "output_audio_s": sum(c.numel() for c in chunks) / 16000.0,
            "source_state_builds": getattr(mono, "source_state_builds", None),
            "e2e": {"value": st.wall_s / audio_s, "unit": "s wall / s audio", "h2d_bytes_per_step": wave.numel() * 4,
                    "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=12, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="s2st", choices=sorted(CONFIGS) + ["stream"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-only", action="store_true", help="one device-resident step only (for ncu launch lists)")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("SB_LANES", "4")),
                    help="batches in flight per GPU (parallel.LanePool: one host thread + stream + search state each); 1 = serial")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.config == "stream":
            print(json.dumps({"impl": "reference", "unavailable": "the streaming agents need SimulEval + fairseq2 (absent offline); "
                                                                   "no CPU port of the streaming chain exists"}))
            return
        run_reference(args, rank)
        return
    if args.config == "stream":
        if rank == 0:
            torch.cuda.set_device(local)
            run_stream(args, torch.device("cuda", local))
        return
    import torch.distributed as dist

    from seamless_communication_b200 import ops, synthetic as S
    from seamless_communication_b200.inference import SequenceGeneratorOptions
    from seamless_communication_b200.parallel import LanePool, OverlappedExchange

    cfg = CONFIGS[args.config]
    BATCH, task = cfg["batch"], cfg["task"]
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    tr = build_models(device)
    eng = tr.model.engine
    opts = SequenceGeneratorOptions(beam_size=BEAM, soft_max_seq_len=(1, 200), hard_max_seq_len=HARD_MAX)
    waves_dev = S.make_waveforms(BATCH, SAMPLES, seed=1234 + rank).to(device)

    def step_device():
        src = tr.fbank_batch(waves_dev)
        return tr.predict(src, task, TGT_LANG, text_generation_opts=opts)

    def launches_now():
        return ops.launch_count() + eng.graph_kernels

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    if args.profile_only:
        step_device()
        torch.cuda.synchronize()
        print(json.dumps({"profile_only": True, "launches": launches_now()}))
        return

    LANES = max(1, args.lanes)
    pool = LanePool(device, LANES, [eng]) if LANES > 1 else None
    main_stream = torch.cuda.current_stream()

    def run_device_steps(n):
        """n steps, each one batch through the whole path; with lanes, LANES of them are in flight at any time.
        Returns what the last step returned."""
        if pool is None:
            for _ in range(n):
                out = step_device()
            return out
        futs = [pool.submit(i, step_device) for i in range(n)]
        for f in futs:
            out, done = f.result()
            main_stream.wait_event(done)
        return out

    # ---- device-resident leg
    if pool is not None:
        pool.warm(step_device)  # one lane at a time: first use captures that lane's step graphs
    run_device_steps(max(args.warmup, LANES))
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    n0 = launches_now()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    last = run_device_steps(args.steps)
    e1.record()
    sync_all()
    ms_dev = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    launches_total = launches_now() - n0  # kernels of this library launched inside the timed region (graph replays included)
    launches = launches_total // args.steps
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        texts, speech = last
        dump_outputs(args.dump_outputs, texts=texts, units=speech.units if speech is not None else None,
                     wavs=speech.audio_wavs if speech is not None else None)

    # one batch at a time (no lanes): the latency of a step and the reference point for the lanes' gain
    step_device()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        step_device()
    e1.record()
    torch.cuda.synchronize()
    ms_serial = max_over_ranks(e0.elapsed_time(e1) / 3)

    # ---- end-to-end leg: host buffers in, host buffers out, copies / collectives overlapped with neighbouring steps
    host_global = None
    if rank == 0:
        host_global = torch.cat([S.make_waveforms(BATCH, SAMPLES, seed=1234 + r) for r in range(world)]).pin_memory()
    max_out = 320 * 512 if task == "s2st" else 0
    xch = OverlappedExchange(BATCH, SAMPLES, max_out, device, world, rank, slots=LANES + 2)

    def consume(w):
        src = tr.fbank_batch(w)
        texts, speech = tr.predict(src, task, TGT_LANG, text_generation_opts=opts)
        return texts, speech

    def publish(speech):
        xch.publish(speech.audio_wavs if speech is not None else None, speech.units if speech is not None else None)

    def e2e_loop(steps):
        # the exchange (PCIe copies, NCCL scatter / gather) stays on this thread so that every rank issues its collectives
        # in the same order; the lanes only compute
        xch.prefetch(host_global)
        if pool is None:
            for i in range(steps):
                w = xch.take()
                if i + 1 < steps:
                    xch.prefetch(host_global)
                publish(consume(w)[1])
        else:
            pending = []

            def finish():
                fut, k = pending.pop(0)
                (_, speech), done = fut.result()
                main_stream.wait_event(done)
                xch.release(k, done)
                publish(speech)

            for i in range(steps):
                w, ready, k = xch.take_async()
                if i + 1 < steps:
                    xch.prefetch(host_global)
                pending.append((pool.submit(i, consume, w, after=ready), k))
                if len(pending) >= LANES:
                    finish()
            while pending:
                finish()
        xch.drain()

    e2e_loop(max(2, LANES))  # warm-up (allocator, graphs for this stream layout)
    sync_all()
    torch.cuda.synchronize()
    e0.record()
    e2e_loop(args.steps)
    e1.record()
    sync_all()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1) / args.steps)

    value = world * BATCH / (ms_dev * 1e-3)
    e2e_value = world * BATCH / (ms_e2e * 1e-3)
    if rank == 0:
        pk = peaks()
        line = {
            "metric": cfg["metric"], "value": value, "unit": "utt/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": workload_config(cfg, BATCH, world),
            "pipeline": {"in_flight": LANES,
                         "lanes": (f"{LANES} batches of {BATCH} in flight per GPU, each on its own stream with its own search state "
                                   "(parallel.LanePool); a step is one batch through the whole path, ms_per_step = time of the K steps / K"
                                   if LANES > 1 else "one batch at a time"),
                         "decoder_step": "persistent kernel" if eng.decode_fused else "launch chain in a CUDA graph"},
            "rtf": ms_dev * 1e-3 / (10.0 * BATCH),
            "serial": {"ms_per_step": ms_serial, "value": world * BATCH / (ms_serial * 1e-3), "unit": "utt/s",
                       "what": "the same step with one batch in flight (latency of a batch; SB_LANES=1 makes this the headline)"},
            "e2e": {"value": e2e_value, "unit": "utt/s", "h2d_bytes_per_step": xch.h2d_bytes, "d2h_bytes_per_step": xch.d2h_bytes,
                    "ms_per_step": ms_e2e, "overlap": "inputs of later steps and outputs of earlier steps move on side streams (exchange on the main thread, compute on the lanes)"},
            "gpu_launches": int(launches_total), "gpu_launches_per_step": int(launches),
            "clocks": clocks,
        }
        if world == 1:
            # two extra (untimed) steps split into stages; where the step goes and each stage against its own bound
            stage_times(tr, waves_dev, task)
            stages = stage_times(tr, waves_dev, task)
            tab = stage_table(stages, BATCH, pk, eng, task)
            line["stages_ms"] = stages
            line["stages"] = tab
            bs = tab["beam_search"]
            tm = measured_decode_traffic() if task == "s2st" else {}
            tsel = tm.get("warm") or tm.get("cold")
            traffic = tsel["dram_bytes_per_step"] if tsel else None
            tsrc = None
            if tsel:
                alg_prof, _ = decode_step_bytes(eng, BATCH, tsel["steps_profiled"])
                tsrc = (f"ncu dram__bytes_read.sum + dram__bytes_write.sum over the launches of a {tsel['steps_profiled']}-step search, per step "
                        f"({'--cache-control none' if 'warm' in tm else 'caches flushed per launch'}; profiles/r02warm_kernels_ncu.txt, "
                        f"profiles/r02_kernels_ncu.txt); algorithmic bytes at those positions: {alg_prof / 1e9:.2f} GB + 0.16 GB of fp32 "
                        f"logits the step also writes; the search's K/V reads grow with the position")
            line["roofline"] = {"bound": "hbm", "kernel": "one beam-search step = decoder-step kernels + vocabulary projection + top-K "
                                                          f"({bs['steps']} steps, {100 * bs['ms'] / ms_serial:.0f} % of a batch's time)",
                                "achieved": bs["achieved_gbs"], "peak": pk["hbm"], "unit": "GB/s", "frac": bs["frac"],
                                "traffic": traffic, "traffic_cold": (tm.get("cold") or {}).get("dram_bytes_per_step"),
                                "traffic_source": tsrc, "algorithmic_bytes": bs["algorithmic_bytes_per_step"],
                                "ms_per_launch_group": bs["ms_per_step"], "peak_source": pk["src"], "in_flight": 1}
            if pool is not None:
                # how the step actually runs: LANES searches interleaved on the device.  Every lane's step still needs every
                # weight once (algorithmic bytes per step unchanged); the effective duration of a step is the time in which
                # LANES searches complete / (LANES x steps)
                enc_res, _ = eng.encode_speech(tr.fbank_batch(waves_dev)["seqs"], None)
                ms_l = lanes_search_ms(pool, eng, enc_res, LANES)
                eff_ms = ms_l / (LANES * bs["steps"])
                ach = bs["algorithmic_bytes_per_step"] / (eff_ms * 1e-3) / 1e9
                line["roofline"].update({"serial": {"achieved": bs["achieved_gbs"], "frac": bs["frac"], "ms_per_launch_group": bs["ms_per_step"]},
                                         "achieved": ach, "frac": ach / pk["hbm"], "ms_per_launch_group": eff_ms, "in_flight": LANES,
                                         "lanes_search_ms": ms_l,
                                         "note": f"{LANES} searches in flight: {ms_l:.1f} ms for {LANES} x {bs['steps']} steps "
                                                 f"(one search alone: {bs['ms']:.1f} ms)"})
        else:
            line["roofline"] = None
        if not args.no_cpu_baseline and world == 1:
            block, ref = cpu_baseline_block(task, 4, 1, warmup=True)
            line["cpu_baseline"] = block
            try:
                line["parity"] = parity_block(tr, ref, waves_dev, task)
            except Exception as ex:  # the bench line must survive a parity failure and show it
                line["parity"] = {"error": repr(ex)}
        print(json.dumps(line), flush=True)
    if pool is not None:
        pool.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
