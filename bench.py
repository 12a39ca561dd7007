#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json: "image-encode ms + decode tokens/s, 7B q4_1").

A *step* = one pass of the hot path over one synthetic batch: encode one 224x224 image (ViT-g + Q-Former + projection),
feed the 32 embedding rows as the image prefix, then generate 128 tokens greedily (BASELINE configs[1]: "Vicuna-7B q4_1
decode-only, 32-token image prefix + 128 generated tokens").  Reported per JSON line:
  value      decode tokens/s with everything resident in HBM (device-chained greedy loop, CUDA-event timed)
  e2e        the same metric through the reference-facing C ABI (minigpt4_encode_image / minigpt4_begin_chat_image /
             128 x minigpt4_end_chat_image) with HOST buffers; host<->device copies and per-token sync inside the timing
  encode_ms  image-encode latency (device, CUDA events) and encode_e2e_ms (wall clock through the ABI)
  roofline   decode dequant-matvec family: algorithmic weight bytes / CUDA-event time per launch vs MEASURED_PEAKS hbm_gbs
  cpu_baseline  the CPU oracle (a restatement of the reference's ggml path) on this box's host cores, bounded sample
`--impl reference` times that CPU path alone (the reference itself cannot be built here: DESIGN.md "Oracle").
N > 1 (torchrun): default --mode replicas = one independent decode stream per GPU (the path is per-session work; no data-path
collective; "scaling": "weak"); --mode tp = the optional tensor-parallel LLaMA step of north_star ("strong").
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_PREFIX, N_GEN = 32, 128
PROMPT = "what is in this picture?"
REF_TOKENS = 32   # decode tokens per step of the CPU arm (bounded sample of the 128-token workload; = north_star's 32-token parity window)


def metric_name(size: str, wtype: str) -> str:
    """ONE string for both arms: the driver only divides the two values when metric / unit / direction are identical."""
    return f"decode tokens/s (Vicuna-{size.upper()} {wtype}, {N_PREFIX}-row image prefix + {N_GEN} generated tokens) + image-encode ms"


def workload(size: str, wtype: str, blocks: int) -> str:
    return (f"configs[{1 if (size, wtype, N_GEN) == ('7b', 'q4_1', 128) else 2 if (size, wtype) == ('7b', 'q5_k') else 3 if (size, wtype) == ('13b', 'q5_k') else '-'}]: Vicuna-{size} {wtype} decode-only, {N_PREFIX}-row image prefix + {N_GEN} generated tokens; "
            f"plus ViT-g f16 224x224 encode ({blocks} blocks) per step")


def dram_ceiling_tok_s(bytes_per_token: float) -> dict:
    """BASELINE.md §3: a CPU decode cannot beat host DRAM bandwidth / weight bytes per token.  Measured with a threaded numpy copy."""
    from oracle import oracle as orc
    n = host_cpus()
    gbs = float(orc.lib().oracle_host_read_gbs(2 << 30, n, 3))
    return {"host_read_gbs": round(gbs, 1), "decode_ceiling_tok_s": round(gbs * 1e9 / bytes_per_token, 2), "how": f"{n}-thread AVX2 read of a 2 GiB buffer, best of 3 (oracle_host_read_gbs)"}


def model_dir() -> Path:
    name = f"minigpt4_b200_models-{os.getuid()}"   # per account: a directory another user created is not writable here
    for cand in ("/dev/shm", "/tmp"):
        try:
            if shutil.disk_usage(cand).free > 12 << 30:
                d = Path(cand) / name
                d.mkdir(parents=True, exist_ok=True)
                return d
        except OSError:
            pass
    d = Path("/tmp") / name
    d.mkdir(parents=True, exist_ok=True)
    return d


def ensure_models(size: str, wtype: str, blocks: int):
    from minigpt4_cpp_b200 import modelgen as mg
    d = model_dir()
    dims = mg.LLAMA_7B if size == "7b" else mg.LLAMA_13B
    llm = d / f"llama-{size}-{wtype}.bin"
    vis = d / f"minigpt4-{size}-f16-b{blocks}.bin"
    info = d / f"llama-{size}-{wtype}.json"
    def part(p):   # (files appear under their final name only when complete)
        return p.with_name(p.name + f".part{os.getpid()}")
    if not (llm.exists() and info.exists()):
        st = mg.write_llama_ggjt(part(llm), mg.LlamaSpec(wtype=wtype, **dims))
        os.replace(part(llm), llm)
        info.write_text(json.dumps(st))
    if not vis.exists():
        mg.write_minigpt4(part(vis), mg.VisionSpec(n_blocks=blocks, n_embd_llm=dims["n_embd"], fast=True))
        os.replace(part(vis), vis)
    return str(vis), str(llm), json.loads(info.read_text())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel: str):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (dram__bytes_read.sum +
    dram__bytes_write.sum; profiles/traffic.json, written from the .ncu-rep of the same build), or None."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        return float(json.loads(p.read_text())[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def host_cpus() -> int:
    """CPUs this process may actually use: affinity mask capped by the cgroup quota (a container often sees 128 logical
    CPUs but is throttled to far fewer; oversubscribing OpenMP threads there is catastrophic)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def pick_threads(llm: str) -> tuple[int, dict]:
    """Give the CPU arm 'all the host threads it can use': time one decode token per candidate thread count, keep the best."""
    from oracle import oracle as orc
    n = host_cpus()
    cands = sorted({c for c in (8, 16, 32, 48, 64, 96, n) if c <= n} | {n})
    e = orc.OracleEngine(None, llm, n_ctx=64, n_threads=cands[0])
    emb = np.random.default_rng(1).standard_normal((2, e.n_embd)).astype(np.float32)
    e.eval_embd(emb)  # touches every weight page once
    timing = {}
    for c in cands:
        e.n_threads = c
        e.end_chat_greedy()
        t0 = time.perf_counter(); e.end_chat_greedy(); timing[c] = time.perf_counter() - t0
        if timing[c] > 20:  # hopeless configuration, stop probing larger counts
            break
    best = min(timing, key=timing.get)
    return best, {str(k): round(v, 4) for k, v in timing.items()}


def cpu_leg(vis: str, llm: str, n_tokens: int, do_encode: bool, threads: int):
    """Time the CPU oracle (restated reference ggml path) on a bounded sample; returns dict + generated ids."""
    from oracle import oracle as orc
    from minigpt4_cpp_b200 import modelgen as mg
    e = orc.OracleEngine(vis if do_encode else None, llm, n_ctx=512, n_threads=threads)
    out = {"cores": threads, "kind": "port"}
    if do_encode:
        img = mg.synth_image()
        t0 = time.perf_counter(); emb = e.encode_image(img); out["encode_ms"] = (time.perf_counter() - t0) * 1e3
    else:
        emb = np.random.default_rng(0).standard_normal((N_PREFIX, e.n_embd)).astype(np.float32)
    t0 = time.perf_counter(); e.eval_embd(emb); out["prefix_ms"] = (time.perf_counter() - t0) * 1e3
    ids = []
    t0 = time.perf_counter()
    for _ in range(n_tokens):
        ids.append(e.end_chat_greedy()[0])
    dt = time.perf_counter() - t0
    out["value"] = n_tokens / dt
    out["unit"] = "tokens/s"
    out["sample"] = f"{n_tokens} greedy decode tokens after the {N_PREFIX}-row image prefix" + (", 1 image encode" if do_encode else "") + ", same synthetic weights"
    return out, ids, emb


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port, all host threads; same metric / config as the GPU arm,
    each step a bounded sample (REF_TOKENS decode tokens; the image encode in the first warm-up and the first timed step)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vis, llm, info = ensure_models(args.size, args.wtype, args.blocks)
    threads, thread_probe = pick_threads(llm)
    from oracle import oracle as orc
    from minigpt4_cpp_b200 import modelgen as mg
    e = orc.OracleEngine(vis, llm, n_ctx=512, n_threads=threads)
    img = mg.synth_image()
    n_tok = args.cpu_tokens or REF_TOKENS
    enc_ms, pre_ms, dec_s, step_s = [], [], [], []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        e.reset_chat()
        encoded = it == 0 or it == args.warmup or args.cpu_encode_every_step
        emb = e.encode_image(img) if encoded else emb
        t1 = time.perf_counter()
        e.eval_embd(emb)
        t2 = time.perf_counter()
        for _ in range(n_tok):
            e.end_chat_greedy()
        t3 = time.perf_counter()
        if it >= args.warmup:
            if encoded: enc_ms.append((t1 - t0) * 1e3)
            pre_ms.append((t2 - t1) * 1e3); dec_s.append(t3 - t2); step_s.append(t3 - t0)
    v = n_tok * len(dec_s) / sum(dec_s)
    bpt = float(info.get("bytes_per_token", 0)) or 4129423360.0
    line = {"impl": "reference", "metric": metric_name(args.size, args.wtype), "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(step_s) / len(step_s), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int8 x int4 dot (Q8_1 x Q4_1), f32 accumulate", "data": "synthetic",
            "config": {"workload": workload(args.size, args.wtype, args.blocks)},
            "encode_ms": max(enc_ms) if enc_ms else None, "prefix_ms": float(np.mean(pre_ms)),
            "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": threads, "kind": "port", "host_cpus": host_cpus(), "thread_probe_s_per_token": thread_probe,
                             "sample": f"{len(dec_s)} steps x {n_tok} greedy decode tokens after the {N_PREFIX}-row prefix (bounded sample of the {N_GEN}-token workload; the rate is "
                                       "position-independent at these lengths); CPU oracle = restatement of ggml@master-31cfbb1 semantics (reference unbuildable offline)",
                             "dram_ceiling": dram_ceiling_tok_s(bpt)},
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def encode_batch8(ext, ctx, mg):
    """BASELINE configs[4], first half: 8 images through minigpt4_b200_encode_images (host buffers in and out, wall clock), next to 8 single calls"""
    imgs = [mg.synth_image(s) for s in range(8)]
    ext.encode_batch(ctx, imgs)                       # builds the lanes (graphs) once
    t = [ext.encode_batch(ctx, imgs)[1] for _ in range(3)]
    t0 = time.perf_counter()
    for im in imgs: ext.encode_array(ctx, im)
    seq = (time.perf_counter() - t0) * 1e3
    return {"images": 8, "wall_ms": min(t), "ms_per_image": min(t) / 8, "sequential_single_calls_ms": seq, "how": "8 concurrent encode lanes (own activations / graph / stream, shared F16 weights)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", default="7b", choices=["7b", "13b"])
    ap.add_argument("--wtype", default="q4_1")
    ap.add_argument("--blocks", type=int, default=39)
    ap.add_argument("--tokens", type=int, default=128, help="generated tokens per step (BASELINE configs[1]: 128; configs[2]: 256)")
    ap.add_argument("--cpu-tokens", type=int, default=0, help="decode tokens of the CPU legs (default: 32)")
    ap.add_argument("--cpu-encode-every-step", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (image embedding, chat reply, "
                                                          "greedy ids, last logits) as DIR/<name>.npy, float32 / float64; the inputs are seeded, "
                                                          "so two builds can be compared output for output")
    ap.add_argument("--mode", default="replicas", choices=["replicas", "tp"],
                    help="N>1: 'replicas' = one independent decode stream per GPU, no data-path collective (weak scaling, default); "
                         "'tp' = one stream, LLaMA layers tensor-parallel over the GPUs with an NCCL sum per row-split matmul (strong scaling)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: --impl ours only")
    global N_GEN
    N_GEN = args.tokens
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    import minigpt4_cpp_b200 as m
    from minigpt4_cpp_b200 import modelgen as mg
    lib = m.load_library()
    ext = m.B200(lib)
    assert ext.L.minigpt4_b200_device_count() > 0, "bench.py needs a CUDA device: the engine has no CPU path"
    ext.L.minigpt4_b200_set_device(local)
    dist = None

    def tp_configure(on: bool):
        """engine contexts loaded after this call are tensor-parallel over all ranks (NCCL id from rank 0) / single-GPU again"""
        import torch
        uid = np.zeros(128, np.uint8)
        if on:
            if rank == 0:
                ext.L.minigpt4_b200_tp_unique_id(uid.ctypes.data_as(ctypes.c_void_p))
            t = torch.from_numpy(uid).cuda(); dist.broadcast(t, 0); uid = t.cpu().numpy()
        ext.L.minigpt4_b200_tp_configure(rank if on else 0, world if on else 1, uid.ctypes.data_as(ctypes.c_void_p))

    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        if args.mode == "tp":
            tp_configure(True)
    if rank == 0:
        paths = ensure_models(args.size, args.wtype, args.blocks)
    if dist:
        dist.barrier()
    vis, llm, info = ensure_models(args.size, args.wtype, args.blocks)

    ctx = lib.minigpt4_model_load(vis, llm, 1, 1337, 2048, 512, 0)
    assert ctx.ptr, "model load failed"
    img = mg.synth_image()
    mi = m.MiniGPT4Image(img.ctypes.data_as(ctypes.c_void_p), 224, 224, 3, m.ImageFormat.F32)

    def barrier():
        if dist:
            import torch
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()

    def step(timed: bool, keep_embedding: bool = False):
        """returns dict: encode_dev_ms, chain_ms, turn_s (whole turn through the ABI), ttft_s, decode_s, ids (+ a copy of the image embedding)"""
        # -- e2e leg: ONE chat turn through the reference ABI with host buffers, wall clock around all of it:
        #    image H2D + encode + embedding D2H | system prompt | embedding H2D + prefix + prompt | 128 x (decode step + 4-byte D2H + id_to_token)
        lib.minigpt4_reset_chat(ctx)
        t0 = time.perf_counter()
        emb = lib.minigpt4_encode_image(ctx, mi)
        t_enc = time.perf_counter()
        enc_dev = ext.stats(ctx).last_encode_ms
        lib.minigpt4_system_prompt(ctx)
        lib.minigpt4_begin_chat_image(ctx, emb, PROMPT)
        t_pre = time.perf_counter()
        toks = [lib.minigpt4_end_chat_image(ctx, temp=0.0)]
        t_first = time.perf_counter()
        toks += [lib.minigpt4_end_chat_image(ctx, temp=0.0) for _ in range(N_GEN - 1)]
        t_end = time.perf_counter()
        # -- device-resident leg: 32-row prefix, then 128 greedy steps chained on the device (no host round trip)
        lib.minigpt4_reset_chat(ctx)
        rows = np.ctypeslib.as_array(emb.data, shape=(emb.n_embeddings,)).reshape(32, -1)
        tp0 = time.perf_counter(); ext.eval_embd(ctx, rows); ext.flush(ctx); prefix_ms = (time.perf_counter() - tp0) * 1e3
        ids, chain_ms = ext.decode_chain(ctx, N_GEN)
        kept = rows.copy() if keep_embedding else None
        lib.minigpt4_free_embedding(emb)
        return {"enc_dev": enc_dev, "enc_wall": (t_enc - t0) * 1e3, "chain_ms": chain_ms, "turn_s": t_end - t0, "ttft_s": t_first - t0,
                "prefill_s": t_pre - t_enc, "decode_s": t_end - t_pre, "prefix_ms": prefix_ms, "ids": ids, "toks": toks, "emb": kept}

    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(local)
    launches0 = ext.stats(ctx).kernel_launches
    barrier()
    sampler.start()
    t_begin = time.perf_counter()
    res = [step(True, keep_embedding=bool(args.dump_outputs) and i == args.steps - 1) for i in range(args.steps)]
    barrier()
    wall = time.perf_counter() - t_begin
    clocks = sampler.stop()
    launches = ext.stats(ctx).kernel_launches - launches0
    if args.dump_outputs and rank == 0:
        # what the last timed step handed its caller, read before anything else runs on the context
        out = Path(args.dump_outputs)
        out.mkdir(parents=True, exist_ok=True)
        last = res[-1]
        np.save(out / "image_embedding.npy", last["emb"].astype(np.float32))                       # minigpt4_encode_image, [32, n_embd]
        np.save(out / "chat_reply_codepoints.npy", np.array([ord(c) for c in "".join(last["toks"])], np.float64))  # N_GEN x minigpt4_end_chat_image
        np.save(out / "decode_ids.npy", last["ids"].astype(np.float64))                            # device-chained greedy ids, [N_GEN]
        np.save(out / "decode_logits.npy", ext.logits(ctx).astype(np.float32))                     # logits of the last chained step, [n_vocab]

    chain_ms = sum(r["chain_ms"] for r in res); turn_s = sum(r["turn_s"] for r in res); dec_s = sum(r["decode_s"] for r in res)
    enc_dev = float(np.mean([r["enc_dev"] for r in res])); enc_wall = float(np.mean([r["enc_wall"] for r in res]))
    ttft_ms = float(np.mean([r["ttft_s"] for r in res])) * 1e3; prefill_ms = float(np.mean([r["prefill_s"] for r in res])) * 1e3
    prefix_ms = float(np.mean([r["prefix_ms"] for r in res]))
    if dist:
        import torch
        t = torch.tensor([chain_ms, turn_s, wall, enc_dev, enc_wall, dec_s, ttft_ms, prefill_ms, prefix_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        chain_ms, turn_s, wall, enc_dev, enc_wall, dec_s, ttft_ms, prefill_ms, prefix_ms = t.tolist()
    streams = world if (world > 1 and args.mode == "replicas") else 1  # independent decode streams in the job
    value = streams * args.steps * N_GEN / (chain_ms * 1e-3)   # whole-job tokens/s: all streams / slowest rank's time
    e2e = streams * args.steps * N_GEN / turn_s                # the same tokens over the WHOLE turn (encode + prompts + prefix + decode, wall clock)
    e2e_decode = streams * args.steps * N_GEN / dec_s          # ... and over the decode calls alone

    # roofline of the decode dequant-matvec family (CUDA events, cold weights: each launch streams a different layer)
    st = ext.stats(ctx)
    peak, peak_src = measured_peaks()
    if st.decode_megakernel:
        # the decode step IS one kernel (decode_megakernel, one launch per token): algorithmic bytes per launch = weight bytes
        # streamed per token; launch duration = CUDA-event time of the chained loop / launches (includes the in-kernel attention,
        # grid barriers and activation staging — nothing is hidden)
        us = chain_ms * 1e3 / (args.steps * N_GEN)  # per launch on one GPU (max over ranks)
        ach = st.llm_weight_bytes_per_token / us * 1e-3
        roofline = {"bound": "hbm", "kernel": f"decode_megakernel<{args.wtype}> (1 launch per token: {st.n_layer} x [qkv, attention, wo, gate_up, down] + output/arg-max)",
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": measured_traffic(f"decode_megakernel_{args.size}_{args.wtype}"), "peak_source": peak_src,
                    "bytes_per_launch": st.llm_weight_bytes_per_token, "us_per_launch": us}
    else:
        kinds = ["qkv", "wo", "gate_up", "down", "output"]
        per_kind, tot_bytes, tot_ms = {}, 0.0, 0.0
        for k, name in enumerate(kinds):
            ms, nb = ext.time_matvec(ctx, k, 3)
            n_launch = 1 if k == 4 else st.n_layer
            per_kind[name] = {"bytes": nb, "us": ms * 1e3, "gbs": nb / ms * 1e-6, "frac": nb / ms * 1e-6 / peak}
            tot_bytes += nb * n_launch; tot_ms += ms * n_launch
        roofline = {"bound": "hbm", "kernel": f"stage_kernel + matvec_kernel<{args.wtype},NT=1> (qkv/wo/gate_up/down x{st.n_layer} + output per token)",
                    "achieved": tot_bytes / tot_ms * 1e-6, "peak": peak, "unit": "GB/s", "frac": tot_bytes / tot_ms * 1e-6 / peak,
                    "traffic": None, "peak_source": peak_src, "bytes_per_token": st.llm_weight_bytes_per_token, "per_kernel": per_kind,
                    "step_effective_gbs": st.llm_weight_bytes_per_token * value * 1e-9}

    n_prompt = len(ext.tokenize(ctx, PROMPT)) if hasattr(ext, "tokenize") else 0
    line = {"metric": metric_name(args.size, args.wtype), "value": value, "unit": "tokens/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall * 1e3 / args.steps, "higher_is_better": True,
            "scaling": "weak" if streams > 1 or world == 1 else "strong", "vs_baseline": None,
            "dtype": "int8 x int4 dot (Q8_1 x Q4_1) f32-accumulate decode and prefill (tcgen05 kind::i8); f16 x f16 -> f32 tcgen05 encode", "data": "synthetic",
            "config": {"workload": workload(args.size, args.wtype, args.blocks),
                       "parallelism": (f"tp{world}" if args.mode == "tp" else f"dp{world} (one independent stream per GPU, no data-path collective)") if world > 1 else "single-gpu", "l2": "inputs larger than L2 (4.1 GB of weights streamed per token vs 126 MB L2)",
                       "value_region": "CUDA-event time of the 128-step device-chained greedy decode loop", "n_ctx": 2048},
            "encode_ms": enc_dev, "encode_e2e_ms": enc_wall, "prefix_ms": prefix_ms,
            "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": int(img.nbytes + 32 * st.n_embd * 4 + 4 * 256), "d2h_bytes_per_step": int(32 * st.n_embd * 4 + 4 * N_GEN),
                    "region": "wall clock of one whole chat turn through the reference C ABI (ctypes, host buffers): minigpt4_encode_image (image H2D, encode, embedding D2H) + "
                              "minigpt4_system_prompt + minigpt4_begin_chat_image (embedding H2D, 32-row prefix, prompt) + 128 x minigpt4_end_chat_image(temp=0) (graph launch, sync, 4-byte D2H each); "
                              "value = 128 tokens / that time",
                    "decode_calls_only": e2e_decode, "decode_calls_note": "the first end_chat call also evaluates the queued prompt rows (deferred, merged prefill): per-token host overhead = this minus prefix_ms", "ttft_ms": ttft_ms, "prefill_ms": prefill_ms, "prompt_tokens_incl_system": n_prompt},
            "encode_batch8": encode_batch8(ext, ctx, mg),
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "engine": {"decode_megakernel_generation": int(st.decode_megakernel), "prefill_gemm": int(getattr(st, "prefill_gemm", 0))}}

    # tensor-parallel leg: on by default for the degrees that ran on hardware (2 and 4); MINIGPT4_BENCH_TP=1 forces it for any N, =0 disables it
    tp_env = os.environ.get("MINIGPT4_BENCH_TP")
    tp_leg = world > 1 and (tp_env == "1" or (tp_env != "0" and world in (2, 4)) or args.mode == "tp")
    if world > 1 and not tp_leg and tp_env != "0":
        line["tp"] = {"world": world, "skipped": "tensor parallelism over %d GPUs has not run on hardware yet (2 and 4 have: profiles/r2_bench_*gpu_dp_and_tp.json); "
                                                "MINIGPT4_BENCH_TP=1 measures it" % world}
    if tp_leg:
        # the tensor-parallel LLaMA step of north_star on the same GPUs (strong scaling: ONE stream over all ranks), measured next to the
        # replica number: 32-row prefix + N_GEN chained greedy tokens, CUDA events, max over ranks; parity against this rank's own 1-GPU context
        import torch
        rows = np.random.default_rng(11).standard_normal((N_PREFIX, st.n_embd)).astype(np.float32)
        if args.mode == "tp":
            c1, c_tp = None, ctx
        else:
            tp_configure(True)
            c_tp = ext.llm_load(llm, n_ctx=2048)
            tp_configure(False)
            c1 = ctx
        lib.minigpt4_reset_chat(c_tp)
        ext.eval_embd(c_tp, rows); lg_tp = ext.logits(c_tp)
        ids_tp, _ = ext.decode_chain(c_tp, N_GEN)                      # warm-up pass (also the parity ids)
        tp_ms = []
        for _ in range(max(1, min(3, args.steps))):
            lib.minigpt4_reset_chat(c_tp)
            ext.eval_embd(c_tp, rows); ext.flush(c_tp)
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            _, ms = ext.decode_chain(c_tp, N_GEN); tp_ms.append(ms)
        ar_us, peer = ext.tp_time_allreduce(c_tp, 64)
        t = torch.tensor([sum(tp_ms), ar_us], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tp_total_ms, ar_us = t.tolist()
        st_tp = ext.stats(c_tp)
        fused = bool(st_tp.decode_megakernel)
        tp_rec = {"world": world, "value": len(tp_ms) * N_GEN / (tp_total_ms * 1e-3), "unit": "tokens/s", "scaling": "strong",
                  "ms_per_token": tp_total_ms / (len(tp_ms) * N_GEN),
                  "path": ("decode megakernel with the all-reduce INSIDE the kernel (OP_REDUCE: flag stores to the peers, partial sums read straight out of peer "
                           "memory over NVLink, 2 per layer)" if fused else
                           "per-op kernels + " + ("one-shot peer-memory all-reduce kernel fused with the residual add (CUDA IPC mappings, loads over NVLink)" if peer
                                                  else "ncclAllReduce + add kernel") + ", 2 per layer"),
                  "standalone_allreduce_us": ar_us, "allreduces_per_token": 2 * st.n_layer,
                  "weight_bytes_per_token_per_gpu": st_tp.llm_weight_bytes_per_token,
                  "hbm_roofline_frac_per_gpu": st_tp.llm_weight_bytes_per_token / (tp_total_ms / (len(tp_ms) * N_GEN) * 1e-3) * 1e-9 / peak}
        if c1 is not None:   # parity of TP against the 1-GPU engine on identical inputs (float order of the partial sums differs: tolerance, not bits)
            lib.minigpt4_reset_chat(c1)
            ext.eval_embd(c1, rows); lg1 = ext.logits(c1)
            ids1, _ = ext.decode_chain(c1, N_GEN)
            n_same = next((i for i, (a, b) in enumerate(zip(ids_tp.tolist(), ids1.tolist())) if a != b), N_GEN)
            tp_rec["parity_vs_1gpu"] = {"logits_rel_err_after_prefix": float(np.abs(lg_tp - lg1).max() / np.abs(lg1).max()), "bar": 1e-2,
                                        "leading_greedy_ids_equal": n_same, "of": N_GEN,
                                        "note": "all ranks are bit-identical to each other; against ONE GPU only the float order of the partial sums differs, and this random-weight "
                                                "32-layer model turns a 1e-6 input perturbation into a 1.9e-2 logit change (DESIGN.md 2.1): tools/tp_check.py holds the 1e-2 bar on "
                                                "2- and 4-layer models (32 of 32 ids)"}
            lib.minigpt4_free(c_tp)
        line["tp"] = tp_rec

    if rank == 0 and not args.no_cpu:
        n_cpu = args.cpu_tokens or REF_TOKENS
        threads, probe = pick_threads(llm)
        cpu, cpu_ids, cpu_emb = cpu_leg(vis, llm, n_cpu, True, threads)
        cpu["host_cpus"] = host_cpus(); cpu["thread_probe_s_per_token"] = probe
        cpu["dram_ceiling"] = dram_ceiling_tok_s(float(st.llm_weight_bytes_per_token))
        line["cpu_baseline"] = cpu
        # parity at FULL size: (1) the vision graph at full depth (39 ViT blocks + 12 Q-Former layers) against the CPU leg's embedding;
        # (2) the oracle, fed the GPU's own embedding, must produce bit-identical logits and the same 32 greedy ids
        from oracle import oracle as orc
        e = orc.OracleEngine(None, llm, n_ctx=512, n_threads=threads)
        lib.minigpt4_reset_chat(ctx)
        emb = ext.encode_array(ctx, img)
        vis_err = float(np.abs(emb - cpu_emb).max() / np.abs(cpu_emb).max())
        ext.eval_embd(ctx, emb); e.eval_embd(emb)
        lg, lc = ext.logits(ctx), e.logits.copy()  # copy: the oracle reuses its logits buffer on every eval
        g_ids, c_ids = [], []
        for _ in range(n_cpu):
            t = ext.greedy_id(ctx); g_ids.append(t); ext.eval_tokens(ctx, [t]); c_ids.append(e.end_chat_greedy()[0])
        line["parity"] = {"vision_rel_err_full_depth": vis_err, "vision_blocks": args.blocks, "vision_bar": 1e-2, "logits_rel_err_after_prefix": float(np.abs(lg - lc).max() / np.abs(lc).max()),
                          "logits_bit_identical": bool(np.array_equal(lg, lc)), "greedy_ids_gpu": g_ids, "greedy_ids_cpu": c_ids, "n_ids": n_cpu,
                          "match": g_ids == c_ids and vis_err < 1e-2}
    if rank == 0:
        print(json.dumps(line), flush=True)
    lib.minigpt4_free(ctx)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
