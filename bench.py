"""Headline benchmark: audio-seconds/s of prefill (and TTFT p50) for Ultravox-v0.5-shaped random-init weights
(Whisper-large-v3 encoder + Llama-3.1-8B), synthetic 30 s / 16 kHz clips, batch 1 per GPU, data-parallel replicas.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--preset v0_5_8b] [--secs 30] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one full pass of the hot path over one clip: waveform -> log-mel -> encoder -> projector -> splice -> Llama
prefill -> last-position logits -> argmax (one CUDA-graph replay of libuvx kernels).  `value` is measured with the
waveform already resident in HBM; `e2e` goes through PrefillEngine.run_e2e with a pinned HOST waveform (H2D inside the
timed region, token D2H + sync per step).  Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "audio-sec/s prefill (Llama-3.1-8B, 30s clip) at 1/2/4/8 B200; TTFT p50"
UNIT = "audio-sec/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--preset", default="v0_5_8b")
    ap.add_argument("--secs", type=float, default=30.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true", help="skip the stock-transformers bf16 GPU arm (N=1 only)")
    ap.add_argument("--no-train-record", action="store_true", help="skip the secondary cfg3 (adapter training) record")
    ap.add_argument("--no-decode-record", action="store_true", help="skip the secondary cfg4-style (graphed decode) record")
    ap.add_argument("--decode-tokens", type=int, default=33, help="tokens generated per stream in the decode record")
    ap.add_argument("--train-batch", type=int, default=4, help="clips per GPU of the secondary cfg3 record")
    ap.add_argument("--ttft-iters", type=int, default=200, help="end-to-end iterations behind TTFT p50 / p90 (>= --steps)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="host threads of the CPU arm (0 = sweep and keep the fastest)")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="wall-clock budget of the CPU arm's timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0: last-position logits, greedy token) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def dump_outputs(out_dir, arrays):
    """One float32 / float64 .npy per output, so that two builds run with the same arguments can be compared array by array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu()
        a = a.float() if a.is_floating_point() else a.double()     # integer outputs (token ids < 2**53) are exact in float64
        np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy())


def workload(cfg, secs):
    """Synthetic request of SURVEY.md 8d: 8 text ids + audio placeholders + 5 text ids, start idx 8."""
    import torch
    n = int(round(16000 * secs))
    frames = -(-n // 160)
    n_tok = -(-frames // 16)
    g = torch.Generator().manual_seed(7)
    ids = torch.cat([torch.randint(0, min(cfg.vocab_size, 128000), (8,), generator=g), torch.full((n_tok,), 128009 % cfg.vocab_size),
                     torch.randint(0, min(cfg.vocab_size, 128000), (5,), generator=g)])[None]
    return dict(n=n, frames=frames, n_tok=n_tok, input_ids=ids, start=torch.tensor([8]),
                tok_len=torch.tensor([n_tok], dtype=torch.int32), abs=torch.tensor([1]))


def config_block(args, cfg, wl, n_gpus):
    return {"workload": f"cfg2: Ultravox-v0.5 shapes ({args.preset}: Whisper-large-v3 encoder + Llama-3.1-8B, random-init), "
                        f"{args.secs:g} s 16 kHz synthetic clip prefill, batch 1 per GPU",
            "clip_seconds": args.secs, "llm_tokens": int(wl["input_ids"].shape[1]), "audio_tokens": wl["n_tok"],
            "batch_per_gpu": 1, "parallelism": f"replicas x{n_gpus} (no collective)",
            "l2": "weights streamed per step (17.6 GB) >> 126 MB L2, so every step re-reads HBM; no explicit flush"}


# ----------------------------------------------------------------------------------------------- CPU arm (oracle)
class CpuOracle:
    """The reference's algorithm (fp32 CPU oracle, `oracle/`) at FULL depth on this box's host cores: log-mel -> conv stem ->
    every encoder layer -> projector -> splice -> every LLM layer -> final norm -> last-row lm_head -> argmax.  Nothing is
    extrapolated: one `step()` is one complete prefill of one clip and returns its wall time per stage.

    Weights: `state` = the GPU model's own state dict (bf16 -> fp32 is exact) when the caller wants the oracle's output as the
    CHECK of the GPU result (bench.py's cpu_baseline leg), else seeded random tensors of the same shapes (the `--impl reference`
    arm, which must not need a GPU).  Per-layer weights are distinct allocations (each layer streams its own 0.9 GB from DRAM,
    like the real model) when host RAM allows, else one layer's tensors are shared by all layers (stated in `sample`)."""

    def __init__(self, cfg, wl, state=None, threads=0):
        import numpy as np
        import psutil
        import torch
        from oracle import logmel as ol, model as om
        self.torch, self.om, self.ol, self.np = torch, om, ol, np
        self.cfg, self.wl = cfg, wl
        self.sh = om.shapes_from_config(cfg)
        sh = self.sh
        self.real = state is not None
        need = 4.0 * (sh.enc_layers * (4 * sh.enc_d ** 2 + 2 * sh.enc_d * sh.enc_ffn) +
                      sh.layers * (sh.d * (sh.heads + 2 * sh.kv_heads) * sh.head_dim + sh.heads * sh.head_dim * sh.d + 3 * sh.d * sh.ffn) +
                      2 * sh.vocab * sh.d)
        self.shared_layers = (not self.real) and psutil.virtual_memory().available < need * 1.3 + 8e9
        if self.real:
            self.sd = state
        else:
            g = torch.Generator().manual_seed(42)

            def r(*shape, std=0.02):
                return torch.randn(*shape, generator=g) * std
            d, f, D, F_ = sh.enc_d, sh.enc_ffn, sh.d, sh.ffn
            sd = {"audio_tower.conv1.weight": r(d, sh.n_mels, 3), "audio_tower.conv1.bias": torch.zeros(d),
                  "audio_tower.conv2.weight": r(d, d, 3), "audio_tower.conv2.bias": torch.zeros(d),
                  "audio_tower.embed_positions.weight": r(sh.enc_max_pos, d), "audio_tower.layer_norm.weight": torch.ones(d),
                  "audio_tower.layer_norm.bias": torch.zeros(d)}
            enc0 = {"self_attn.q_proj.weight": r(d, d), "self_attn.k_proj.weight": r(d, d), "self_attn.v_proj.weight": r(d, d),
                    "self_attn.out_proj.weight": r(d, d), "fc1.weight": r(f, d), "fc2.weight": r(d, f),
                    "self_attn.q_proj.bias": torch.zeros(d), "self_attn.v_proj.bias": torch.zeros(d),
                    "self_attn.out_proj.bias": torch.zeros(d), "fc1.bias": torch.zeros(f), "fc2.bias": torch.zeros(d),
                    "self_attn_layer_norm.weight": torch.ones(d), "self_attn_layer_norm.bias": torch.zeros(d),
                    "final_layer_norm.weight": torch.ones(d), "final_layer_norm.bias": torch.zeros(d)}
            llm0 = {"input_layernorm.weight": torch.ones(D), "post_attention_layernorm.weight": torch.ones(D),
                    "self_attn.q_proj.weight": r(sh.heads * sh.head_dim, D), "self_attn.k_proj.weight": r(sh.kv_heads * sh.head_dim, D),
                    "self_attn.v_proj.weight": r(sh.kv_heads * sh.head_dim, D), "self_attn.o_proj.weight": r(D, sh.heads * sh.head_dim),
                    "mlp.gate_proj.weight": r(F_, D), "mlp.up_proj.weight": r(F_, D), "mlp.down_proj.weight": r(D, F_)}
            for i in range(sh.enc_layers):
                for k, v in enc0.items():
                    sd[f"audio_tower.layers.{i}.{k}"] = v if (self.shared_layers or i == 0) else v.clone()
            for i in range(sh.layers):
                for k, v in llm0.items():
                    sd[f"language_model.model.layers.{i}.{k}"] = v if (self.shared_layers or i == 0) else v.clone()
            sd["language_model.model.norm.weight"] = torch.ones(D)
            sd["language_model.model.embed_tokens.weight"] = r(sh.vocab, D)
            sd["language_model.lm_head.weight"] = sd["language_model.model.embed_tokens.weight"] if sh.tie_embeddings else r(sh.vocab, D)
            pj = "multi_modal_projector."
            sd[pj + "ln_pre.weight"] = torch.full((d * sh.stack,), 0.4)
            sd[pj + "linear_1.weight"] = r(sh.proj_hidden, d * sh.stack)
            sd[pj + "ln_mid.weight"] = torch.full((sh.proj_hidden // 2,), 0.4)
            sd[pj + "linear_2.weight"] = r(D, sh.proj_hidden // 2)
            self.sd = sd
        self.threads = threads
        self.sweep = None
        if not threads:
            self.sweep = self._sweep_threads()
            self.threads = min(self.sweep, key=self.sweep.get)
        torch.set_num_threads(self.threads)

    def _sweep_threads(self):
        """One encoder layer + one LLM layer at each thread count; oversubscribing the cores (round 1 used os.cpu_count()
        = 128 hyperthreads) made the same layer 6x slower than at 8-32 threads."""
        torch, om, sh = self.torch, self.om, self.sh
        cores = os.cpu_count() or 1
        cand = sorted({c for c in (8, 16, 32, 64, 96, cores // 2, cores) if 1 <= c <= cores} or {cores})
        h = torch.randn(1, sh.enc_max_pos, sh.enc_d) * 0.1
        S = int(self.wl["input_ids"].shape[1])
        e = torch.randn(1, S, sh.d) * 0.1
        cos, sin = om.rope_cos_sin(sh, torch.arange(S)[None])
        causal = torch.triu(torch.full((S, S), torch.finfo(torch.float32).min), diagonal=1)[None, None]
        out = {}
        with torch.no_grad():
            for c in cand:
                torch.set_num_threads(c)
                best = 1e9
                for rep in range(2):
                    t0 = time.perf_counter()
                    om.whisper_layer(self.sd, "audio_tower.layers.0.", h, None, sh.enc_heads)
                    om.llama_layer(self.sd, "language_model.model.layers.0.", sh, e, cos, sin, causal)
                    best = min(best, time.perf_counter() - t0)
                out[c] = best
        return out

    def step(self, wave, mel_used=None):
        """One full-depth prefill of `wave` (float32 numpy, 16 kHz).  Returns (stage seconds, last-row logits [V], token).
        `mel_used`: the bf16-rounded mel the GPU path consumed (check mode: isolates everything after the front end, which has
        its own parity test against the float64 oracle); the oracle's own mel is still computed and timed."""
        torch, om, ol, sh, wl = self.torch, self.om, self.ol, self.sh, self.wl
        t = {}
        with torch.no_grad():
            t0 = time.perf_counter()
            padded, frames = ol.pad_batch([wave])
            mel = torch.from_numpy(ol.log_mel(padded, sh.n_mels, dtype=self.np.float32))
            t["mel"] = time.perf_counter() - t0
            if mel_used is not None:
                self.mel_max_abs_diff = float((mel - mel_used).abs().max())
                mel = mel_used
            t0 = time.perf_counter()
            enc = om.whisper_encoder(self.sd, sh, mel, torch.tensor([int(frames[0])]))
            t["encoder"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            aud = om.projector(self.sd, sh, enc)
            emb = self.sd["language_model.model.embed_tokens.weight"][wl["input_ids"]].clone()
            om.splice(emb, aud, wl["start"], wl["tok_len"], wl["abs"])
            t["projector_splice"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            logits = om.llama_forward(self.sd, sh, emb, last_only=True).view(-1)
            tok = int(logits.argmax())
            t["llm_prefill_lm_head"] = time.perf_counter() - t0
        t["total"] = sum(t.values())
        return t, logits, tok

    def describe(self, n_steps):
        sh = self.sh
        return (f"fp32 CPU oracle ({'GPU model weights' if self.real else 'seeded random weights'}"
                f"{', one layer shared by all layers (host RAM)' if self.shared_layers else ''}), {n_steps} full prefill(s) of one "
                f"{self.wl['n'] / 16000:g} s clip at FULL depth ({sh.enc_layers} encoder + {sh.layers} LLM layers, last-row lm_head), "
                f"{self.threads} threads" + (f" (sweep s/layer-pair: {({k: round(v, 3) for k, v in self.sweep.items()})})" if self.sweep else ""))


def cpu_leg(cfg, wl, args, state=None, gpu_logits=None, gpu_token=None, max_steps=2, warm=0, mel_used=None, lib_logits=None):
    """cpu_baseline for the main line (1 timed full-depth step on the GPU model's weights, doubling as the output check) or the
    body of the `--impl reference` arm (random weights, up to `max_steps` timed steps inside --cpu-budget-s)."""
    import numpy as np
    orc = CpuOracle(cfg, wl, state, args.cpu_threads)
    wave = np.random.default_rng(1000).standard_normal(wl["n"]).astype(np.float32)
    for _ in range(warm):
        orc.step(wave, mel_used)
    steps, t_begin = [], time.perf_counter()
    logits = tok = None
    while len(steps) < max_steps and (not steps or time.perf_counter() - t_begin + steps[-1]["total"] < args.cpu_budget_s):
        t, logits, tok = orc.step(wave, mel_used)
        steps.append(t)
    best = min(steps, key=lambda d: d["total"])
    secs = wl["n"] / 16000.0
    out = {"value": secs / best["total"], "unit": UNIT, "cores": orc.threads, "kind": "port", "sample": orc.describe(len(steps)),
           "stage_seconds": {k: round(v, 4) for k, v in best.items()}, "ttft_s": best["total"],
           "step_seconds": [round(d["total"], 3) for d in steps], "host_cpus": os.cpu_count()}
    check = None
    if gpu_logits is not None:
        import torch
        g = gpu_logits.float().cpu().view(-1)
        rel = float((g - logits).norm() / logits.norm())
        top5 = logits.topk(5).indices.tolist()
        # SURVEY 7 (ii): end-to-end error against the fp32 oracle is judged against HF's own bf16 forward on the SAME weights and
        # mel (stock transformers modules on this GPU), both numbers side by side; 3e-2 is the bound when that arm did not run
        lib_rel = None
        if lib_logits is not None:
            lib_rel = float((lib_logits.float().view(-1) - logits).norm() / logits.norm())
        bound = max(3e-2, 1.25 * lib_rel) if lib_rel is not None else 3e-2
        check = {"what": "GPU engine's last-row logits / token vs the full-depth fp32 CPU oracle on the same weights and clip",
                 "logits_rel_err": rel, "library_bf16_logits_rel_err_same_weights": lib_rel, "gpu_token": int(gpu_token),
                 "oracle_token": int(tok), "library_token": int(lib_logits.argmax()) if lib_logits is not None else None,
                 "gpu_token_in_oracle_top5": int(gpu_token) in top5,
                 "oracle_logit_gap_of_gpu_token": float(logits.max() - logits[int(gpu_token)]),
                 "mel_max_abs_diff_gpu_vs_oracle": getattr(orc, "mel_max_abs_diff", None),
                 "tolerance": "rel <= max(3e-2, 1.25 x the error of HF's own bf16 forward on the same weights) and the token in the oracle's top-5",
                 "ok": bool(rel <= bound and int(gpu_token) in top5)}
    return out, check


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- roofline pass
def roofline_pass(model, eng, peaks, reps=20):
    """Average launch duration of the dominant kernel - the weight-streaming GEMM of the Llama prefill (M = S = 201 tokens
    against 15 GB of weights: HBM-bound) - measured with CUDA events around CUDA-GRAPH replays that hold exactly the GEMM calls
    of one step (recorded from the engine's own step, same arguments and buffers, back to back like in the real graph), on the
    launching stream, right after the timed region.  Round 1 timed each launch eagerly with its own event pair, which added
    ~25 % of launch gaps to a 30 us kernel.  One "launch" = one uvx_gemm_* call (including its split-K reduce pass, if any).
    Algorithmic bytes per launch = W (N*K*2) + A (M*K*2) + C (M*N*out) (+ residual read); the encoder GEMMs (tensor-bound) are
    measured the same way."""
    import torch
    from ultravox_b200 import ops
    calls = []
    hooks = {}

    def record(name):
        orig = getattr(ops, name)

        def wrapped(*a, **k):
            calls.append((name, orig, a, k))
            return orig(*a, **k)
        hooks[name] = orig
        setattr(ops, name, wrapped)

    for name in ("gemm_raw", "linear_tiled"):
        if hasattr(ops, name):
            record(name)
    try:
        eng._step()
        torch.cuda.synchronize()
    finally:
        for name, orig in hooks.items():
            setattr(ops, name, orig)
    S = eng.input_ids.shape[1] * eng.input_ids.shape[0]

    def shape_of(c):
        name, _, a, k = c
        if name == "gemm_raw":
            M, K, W, C_t = a[1] * a[2], a[3], a[6], a[7]
            R = k.get("R", a[13] if len(a) > 13 else None)
            return M, W.shape[0], K, C_t.element_size(), R is not None
        x, wt = a[0], a[1]                      # ops.linear_tiled(x, TiledWeight, ...): N weight rows, n_out output columns
        rows = x.numel() // x.shape[-1]
        return rows, wt.N, x.shape[-1], 2 * (wt.n_out if k.get("act", 0) == ops.ACT_SWIGLU else wt.N) / wt.N, k.get("residual") is not None

    def group(pred):
        sel = [c for c in calls if pred(*shape_of(c)[:3])]
        if not sel:
            return None
        byt = fl = 0.0
        for c in sel:
            M, N, K, osz, has_r = shape_of(c)
            byt += N * K * 2 + M * K * 2 + M * N * osz + (M * N * 2 if has_r else 0)
            fl += 2.0 * M * N * K
        # manual capture on a side stream: `with torch.cuda.graph()` empties the allocator cache first, which would unmap the
        # (already freed, still cached) activation buffers the recorded calls point at
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g.capture_begin()
            for _, orig, a, k in sel:
                orig(*a, **k)
            g.capture_end()
        torch.cuda.current_stream().wait_stream(side)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3 / reps
        return t, byt, fl, len(sel)

    out = {}
    llm = group(lambda M, N, K: M == S and K >= 2048)
    if llm:
        t, byt, fl, n = llm
        peak = peaks.get("hbm_gbs", 6650.0)
        traffic = None
        for fn in ("r2_traffic.json", "r1_traffic.json"):   # DRAM bytes per launch of the same launches from the committed ncu capture
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", fn)))["dram_bytes_per_launch_avg"]
                break
            except Exception:
                pass
        out = {"bound": "hbm", "kernel": "Llama-prefill weight-streaming GEMM (M=%d), %d launches/step" % (S, n), "achieved": byt / t / 1e9,
               "peak": peak, "unit": "GB/s", "frac": byt / t / 1e9 / peak, "traffic": traffic, "launches": n,
               "avg_launch_us": t / n * 1e6, "bytes_per_launch_avg": byt / n, "all_launches_ms": t * 1e3,
               "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
               "how": "CUDA events around %d replays of a CUDA graph holding one step's %d GEMM calls back to back, launching stream" % (reps, n)}
    enc = group(lambda M, N, K: M > S)
    if enc:
        t, byt, fl, n = enc
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        out["encoder_gemms"] = {"bound": "tensor", "achieved": fl / t / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": fl / t / 1e12 / peak,
                                "launches": n, "avg_launch_us": t / n * 1e6, "all_launches_ms": t * 1e3}
    return out


# ----------------------------------------------------------------------------------------------- cfg3 record
def train_record(model, cfg, args, rank, world, dev):
    """Secondary record (VERDICT r1 item 7): BASELINE config 3 - adapter-only training, encoder + LLM frozen, bf16, data-parallel,
    ONE gradient all-reduce per optimizer step - on the same weights, `--train-batch` 30 s clips per GPU, 1 warm-up + 3 timed
    steps (CUDA events, max over ranks).  The all-reduce is timed separately (events on the launching stream around the NCCL
    call).  This is the only path of the repo with a collective, so it is what the 1 -> 8 GPU scaling run sees of it."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from ultravox_b200 import ops
    from ultravox_b200.training import AdapterTrainer
    B, secs = args.train_batch, args.secs
    n = int(16000 * secs)
    frames = -(-n // 160)
    n_tok = -(-frames // 16)
    g = torch.Generator().manual_seed(7 + rank)
    S = 8 + n_tok + 5
    ids = torch.randint(0, min(cfg.vocab_size, 128000), (B, S), generator=g)
    labels = ids.clone()
    labels[:, :-5] = -100
    waves = np.stack([np.random.default_rng(5000 + rank * 1000 + i).standard_normal(n).astype(np.float32) for i in range(B)])
    waves = torch.from_numpy(np.pad(waves, ((0, 0), (0, (-n) % 160)))).to(dev)
    tr = AdapterTrainer(model, lr=2e-3)
    ar_ms = []

    def step():
        tm = ops.logmel(waves, cfg.audio_config.num_mel_bins, want_f32=False, want_tm=True)
        loss = tr.forward_backward(input_ids=ids, audio_values=None, audio_token_start_idx=torch.full((B,), 8),
                                   audio_lens=torch.full((B,), frames), audio_token_len=torch.full((B,), n_tok, dtype=torch.int32),
                                   audio_batch_size=torch.ones(B, dtype=torch.int64), labels=labels, audio_tm=tm)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        scale = tr.all_reduce()
        a1.record()
        tr.optimizer_step(scale)
        ar_ms.append((a0, a1))
        return loss

    flat0 = model.multi_modal_projector.flat.clone()
    loss0 = float(step())
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ar_ms.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        loss = step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 3, max(a.elapsed_time(b) for a, b in ar_ms)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    loss1 = float(loss)
    model.multi_modal_projector.flat.copy_(flat0)          # leave the weights as the other passes expect them
    # the released recipes' variant (audio_model_lora_config r = 8, SURVEY 8f-3): the same step with LoRA adapters on the encoder's
    # q / k projections trained too - encoder training forward (activations kept) + full encoder backward
    lora_ms = None
    if not getattr(args, "no_train_lora", False):
        try:
            from ultravox_b200.autograd import EncoderLora
            lora = EncoderLora(model, r=8, alpha=8.0, seed=1)
            tr2 = AdapterTrainer(model, lr=2e-3, encoder_lora=lora)
            tr_saved, tr = tr, tr2
            step()
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(2):
                step()
            f1.record()
            torch.cuda.synchronize()
            tl = torch.tensor([f0.elapsed_time(f1) / 2], device=dev)
            if world > 1:
                dist.all_reduce(tl, op=dist.ReduceOp.MAX)
            lora_ms = float(tl[0])
            tr = tr_saved
            lora.unmerge(model)
            model.multi_modal_projector.flat.copy_(flat0)
            del lora, tr2
            torch.cuda.empty_cache()
        except Exception as e:
            lora_ms = "error: " + repr(e)[:200]
    ms, ar = float(t[0]), float(t[1])
    return {"config": "cfg3: adapter-only training (encoder + LLM frozen), bf16, data-parallel, one gradient all-reduce per step",
            "per_gpu_batch": B, "global_batch": B * world, "clip_seconds": secs, "steps": 3, "warmup": 1, "ms_per_step": ms,
            "clips_per_s": B * world / (ms * 1e-3), "audio_sec_per_s": B * world * secs / (ms * 1e-3),
            "with_encoder_lora_r8_ms_per_step": lora_ms,
            "allreduce_ms": ar if world > 1 else 0.0, "allreduce_bytes": tr.grad.numel() * 4 if world > 1 else 0,
            "allreduce": "NCCL sum all-reduce of the flat fp32 projector gradient; 1/world folded into the AdamW kernel" if world > 1 else "none (1 GPU)",
            "loss_first": loss0, "loss_last": loss1, "timer": "CUDA events, max over ranks"}


# ----------------------------------------------------------------------------------------------- main
def decode_record(model, cfg, eng, args, world):
    """Secondary record (BASELINE config 4's serving loop on the cfg2 backbone): prefill of the bench clip's prompt, then
    `--decode-tokens` greedy decode steps, each ONE CUDA-graph replay of `DecodeEngine` (embedding -> 32 layers of weight-streaming
    GEMV / KV-cache attention -> lm head -> pick -> bookkeeping, nothing on the host), for 1 and 8 concurrent streams per GPU.
    CUDA events around the decode loop; the HBM fraction counts the decoder weights once per step (what a step must read)."""
    import torch
    from ultravox_b200.engine import DecodeEngine
    out = {"config": "cfg4 serving loop on the cfg2 (8B) backbone: 30 s clip prefill + greedy decode, CUDA-graphed step; the 70B replica "
                     "is scripts/bench_configs.py decode", "new_tokens": args.decode_tokens, "streams": {}}
    lm = model.language_model
    wbytes = sum(p.numel() for n, p in lm.named_parameters() if "embed_tokens" not in n) * 2
    peak = 0.0
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    from ultravox_b200 import ops
    with torch.no_grad():                                      # the spliced prompt of the bench clip (same stages as the engine's step)
        tm = ops.logmel(eng.wave, eng.n_mels, want_f32=False, want_tm=True)
        aud = model.project_audio(model.encode_audio(tm, None, kv_len=eng.kv_len))
        Bp, Sp = eng.input_ids.shape
        src = ops.splice_plan(eng.start, eng.tok_len, eng.abs, Bp, Sp, aud.shape[1])
        emb1 = ops.embed_splice(eng.input_ids, lm.model.embed_tokens.weight, aud, src)[:1].clone()
    for B in (1, 8):
        emb = emb1.expand(B, -1, -1).contiguous()
        S = emb.shape[1]
        de = DecodeEngine(model, B, S + args.decode_tokens + 2)
        for rep in range(2):                                   # first pass captures the graph
            torch.cuda.synchronize()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            de.prefill(emb.clone())
            e1.record()
            for _ in range(args.decode_tokens - 1):
                de.step()
            e2.record()
            torch.cuda.synchronize()
        ms_tok = e1.elapsed_time(e2) / max(1, args.decode_tokens - 1)
        out["streams"][str(B)] = {"prefill_ms": e0.elapsed_time(e1), "decode_ms_per_token": ms_tok,
                                  "tok_per_s_per_gpu": B / (ms_tok * 1e-3), "tok_per_s_all_gpus": world * B / (ms_tok * 1e-3),
                                  "hbm_frac_weights_once": (wbytes / (ms_tok * 1e-3) / 1e9 / peak) if peak else None,
                                  "launches_per_step": de.launches_per_step}
        del de
        torch.cuda.empty_cache()
    out["weights_gb"] = wbytes / 1e9
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    from ultravox_b200.config import preset
    cfg = preset(args.preset)
    import torch
    wl = workload(cfg, args.secs)

    if args.impl == "reference":
        # the reference's own path is CPU PyTorch (pure Python repo); it cannot be pip-installed/imported here verbatim
        # (accelerate/peft/librosa absent, transformers 4->5 drift; DESIGN.md), so the arm times the oracle port - at FULL depth,
        # every step a complete prefill of one clip; `steps` in the line is what was actually executed inside --cpu-budget-s.
        if rank != 0:
            return
        t0 = time.perf_counter()
        cb, _ = cpu_leg(cfg, wl, args, max_steps=max(1, args.steps), warm=1 if args.warmup > 0 else 0)
        n_done = len(cb["step_seconds"])
        mean_s = sum(cb["step_seconds"]) / n_done
        secs = wl["n"] / 16000.0
        line = {"impl": "reference", "metric": METRIC, "value": secs / mean_s, "unit": UNIT, "n_gpus": args.gpus, "steps": n_done,
                "steps_requested": args.steps, "warmup": 1 if args.warmup > 0 else 0, "ms_per_step": mean_s * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_block(args, cfg, wl, args.gpus),
                "cpu_baseline": {"value": secs / mean_s, **{k: cb[k] for k in ("unit", "cores", "kind", "sample", "stage_seconds", "host_cpus")}},
                "e2e": {"value": secs / mean_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "ttft_ms_p50": statistics.median(cb["step_seconds"]) * 1e3, "step_seconds": cb["step_seconds"],
                "wall_s": time.perf_counter() - t0}
        print(json.dumps(line))
        return

    import numpy as np
    import torch.distributed as dist
    from ultravox_b200 import _lib
    from ultravox_b200.engine import PrefillEngine
    from ultravox_b200.model import UltravoxModel

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    model = UltravoxModel(cfg, device=dev).init_random_(seed=42)
    eng = PrefillEngine(model, wl["n"], wl["input_ids"], wl["start"], wl["tok_len"], wl["abs"])
    K, W = args.steps, max(args.warmup, 3)
    n_wave = min(K, 8)
    host = [torch.from_numpy(np.random.default_rng(1000 + rank * 100 + i).standard_normal(wl["n"]).astype(np.float32))[None]
            for i in range(n_wave)]
    host = [torch.nn.functional.pad(h, (0, eng.L - h.shape[1])).pin_memory() for h in host]
    devw = [h.to(dev) for h in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value")
    for i in range(W):
        eng.wave.copy_(devw[i % n_wave])
        eng.run()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(K):
        eng.wave.copy_(devw[i % n_wave])      # D2D stage of the resident waveform into the graph's input buffer
        eng.run()
    e1.record()
    barrier()
    last_step = {"logits": eng.logits.clone(), "token": eng.token.clone()}    # the later passes overwrite the engine's buffers
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    # ---- end to end through the public engine call with HOST buffers
    for i in range(3):
        eng.run_e2e(host[i % n_wave])
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        eng.run_e2e(host[i % n_wave])
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    # ---- TTFT distribution: >= 200 end-to-end requests regardless of --steps (SURVEY 8d), host clock around a final sync and
    # CUDA events on the compute stream, both reported
    n_tt = max(K, args.ttft_iters)
    per, per_ev = [], []
    for i in range(n_tt):
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0 = time.perf_counter()
        ea.record()
        eng.run_e2e(host[i % n_wave])
        eb.record()
        per.append(time.perf_counter() - s0)
        per_ev.append((ea, eb))
    torch.cuda.synchronize()
    per_ev = sorted(a.elapsed_time(b) for a, b in per_ev)
    per_sorted = sorted(per)

    # ---- output check material: the engine's logits / token for the seed-1000 clip (rank 0 compares with the CPU oracle below)
    eng.run_e2e(host[0])
    gpu_logits, gpu_token = eng.logits.clone(), int(eng.token[0])
    tokens_ok = 0 <= gpu_token < cfg.vocab_size and bool(torch.isfinite(gpu_logits).all())

    train = None
    if not args.no_train_record:
        try:
            train = train_record(model, cfg, args, rank, world, dev)
        except Exception as e:
            train = {"error": repr(e)[:300]}

    decode = None
    if not args.no_decode_record:
        try:
            decode = decode_record(model, cfg, eng, args, world)
        except Exception as e:
            decode = {"error": repr(e)[:300]}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        secs = wl["n"] / 16000.0
        line = {"metric": METRIC, "value": world * K * secs / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic", "config": config_block(args, cfg, wl, world),
                "e2e": {"value": world * K * secs / float(e2e_s), "unit": UNIT, "h2d_bytes_per_step": int(host[0].numel() * 4),
                        "d2h_bytes_per_step": 8, "timer": "host perf_counter around K engine.run_e2e calls, max over ranks"},
                "ttft_ms_p50": statistics.median(per) * 1e3, "ttft_ms_p90": per_sorted[int(0.9 * (len(per) - 1))] * 1e3,
                "ttft_ms_p50_cuda_events": per_ev[len(per_ev) // 2], "ttft_iters": n_tt,
                "gpu_launches": eng.launches_per_step * K, "launches_per_step": eng.launches_per_step,
                "clocks": clocks, "token_check": tokens_ok, "train": train, "decode": decode}
        state = mel_used = lib_logits = None
        if not args.no_cpu_baseline:
            try:      # material for the CPU leg, fetched before anything else touches the allocator
                from ultravox_b200 import ops
                from oracle import model as om
                mel_used = ops.logmel(devw[0], model.audio_tower.n_mels).cpu().to(torch.bfloat16).float()
                state = om.state_dict_fp32(model)
            except Exception as e:
                line["cpu_baseline"] = {"error": repr(e)[:300]}
        if not args.no_roofline:
            try:
                line["roofline"] = roofline_pass(model, eng, peaks)
            except Exception as e:  # never lose the headline number to the diagnostic pass
                line["roofline"] = {"error": repr(e)[:300]}
        if world == 1 and not args.no_library_baseline:
            try:
                sys.path.insert(0, os.path.join(ROOT, "scripts"))
                import hf_gpu_baseline
                lib_out = hf_gpu_baseline.run(cfg, wl, dev, iters=20, warmup=3, state=model.state_dict(), check_mel=mel_used)
                lib_logits = lib_out.pop("_check_logits", None)
                line["gpu_library_baseline"] = lib_out
            except Exception as e:
                line["gpu_library_baseline"] = {"error": repr(e)[:300]}
        if state is not None:
            # full-depth fp32 CPU oracle on THIS model's weights: the cpu_baseline sample and the check of the GPU output in one
            try:
                cb, check = cpu_leg(cfg, wl, args, state=state, gpu_logits=gpu_logits, gpu_token=gpu_token, max_steps=1,
                                    mel_used=mel_used, lib_logits=lib_logits)
                line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "stage_seconds", "host_cpus")}
                line["check"] = check
                line["token_check"] = bool(tokens_ok and check["ok"])
            except Exception as e:      # e.g. host RAM too small for the fp32 copy: keep the headline, say what happened
                line["cpu_baseline"] = {"error": repr(e)[:300]}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
