#!/usr/bin/env python
"""bench.py -- VITA omni forward path on B200: 1 image + 10 s audio + text prefill -> 256-token greedy decode,
Mixtral-8x7B geometry (32 layers, bf16, random-init weights, synthetic inputs).

    python bench.py --gpus 1 --steps K --warmup W              # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                     # + the last timed step's outputs as DIR/<name>.npy
    python bench.py --impl reference --gpus 1 --steps K ...    # the reference algorithm on the host CPU (oracle port)
    torchrun --nproc-per-node N bench.py --gpus N ...          # N independent replicas (request parallel, weak scaling)

A step = one complete generate(): InternViT + Whale encoders, splice, 32-layer sparse-MoE prefill, 256 decode steps.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from vita_b200.config import VitaConfig, IMAGE_TOKEN_INDEX, AUDIO_TOKEN_INDEX  # noqa: E402

METRIC = "omni_generated_tokens_per_s"
UNIT = "tokens/s"
TEXT_TOKENS = 128
AUDIO_FRAMES = 998            # 10 s of 10 ms fbank frames: 1 + (160000 - 400) // 160


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=float(d["hbm_gbs"]), tflops=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback (B200_PROFILING.md)")


def prefill_flops(S: int, cfg) -> float:
    """Algorithmic FLOPs of the Mixtral prefill (SURVEY.md section 8d): GEMMs + causal attention + last-row lm_head."""
    c = cfg.llm
    H, I, L, D = c.hidden_size, c.intermediate_size, c.num_hidden_layers, c.head_dim
    per_tok_layer = 2 * H * (c.qkv_rows) + 2 * H * c.num_attention_heads * D + 2 * H * c.num_local_experts \
        + c.num_experts_per_tok * 3 * 2 * H * I
    attn = 2 * S * S * c.num_attention_heads * D * L   # QK^T + PV, causal-halved
    return per_tok_layer * L * S + attn + 2 * H * c.vocab_size


def decode_bytes(ctx: int, cfg) -> float:
    """Algorithmic HBM bytes of one bs=1 decode step (SURVEY.md section 8d)."""
    c = cfg.llm
    H, I, L, D = c.hidden_size, c.intermediate_size, c.num_hidden_layers, c.head_dim
    per_layer = (c.qkv_rows * H + H * c.num_attention_heads * D) * 2 + c.num_local_experts * H * 2 \
        + c.num_experts_per_tok * 3 * H * I * 2 + 2 * H * 2
    kv = 2 * c.num_key_value_heads * D * 2 * ctx
    return L * (per_layer + kv) + c.vocab_size * H * 2 + H * 2


def encoder_flops(cfg) -> float:
    return 0.723e12 + 17.2e9 + 0.276e12   # InternViT tile + projector + Whale 10 s (SURVEY.md section 8d)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_inputs(cfg, seed=0, pin=True):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, cfg.llm.vocab_size, (1, TEXT_TOKENS), generator=g)
    ids[0, 1] = IMAGE_TOKEN_INDEX
    ids[0, 2] = AUDIO_TOKEN_INDEX
    images = torch.randn(1, 3, cfg.vision.image_size, cfg.vision.image_size, generator=g)
    feats = torch.randn(1, AUDIO_FRAMES, cfg.audio.input_dim, generator=g)
    lengths = torch.tensor([AUDIO_FRAMES])
    if pin and torch.cuda.is_available():
        images, feats = images.pin_memory(), feats.pin_memory()
    return ids, images, feats, lengths


def spliced_len(cfg) -> int:
    t2 = cfg.audio.frames_after_subsampling(AUDIO_FRAMES)
    return TEXT_TOKENS - 2 + cfg.vision.out_tokens + cfg.audio.tokens_after_adapter(t2)


# ================================================================================================ CPU arm (oracle port)
def cpu_reference_state(layers_cpu: int):
    """fp32 weights of the CPU arm: full-size InternViT + Whale + projector, Mixtral at full layer width but
    `layers_cpu` layers (what host RAM and a few minutes allow); values need not match the GPU arm's (timing only)."""
    from vita_b200 import weights as W
    cfg = VitaConfig.full(num_hidden_layers=layers_cpu)
    import zlib
    shapes = W.all_param_shapes(cfg)
    g = torch.Generator().manual_seed(0)
    # timing only: the values need not match the GPU arm's, so the matrices are cut out of one 16 M-entry normal
    # block at a per-tensor offset (host RNG at 1.45 G draws per layer would cost minutes)
    block = (torch.randn(1 << 24, generator=g) * 0.02).bfloat16().float()
    state = {}
    for name, shape in shapes.items():
        if "global_cmvn" in name:
            state[name] = torch.zeros(shape) if name.endswith("mean") else torch.ones(shape)
        elif len(shape) == 1 and ("norm" in name or "bn2" in name or "embed.1" in name) and name.endswith("weight"):
            state[name] = torch.ones(shape)
        elif name.endswith(("ls1", "ls2")):
            state[name] = torch.full(shape, 0.5)
        else:
            n = 1
            for d in shape:
                n *= d
            start = zlib.crc32(name.encode()) % block.numel()
            rolled = torch.cat([block[start:], block[:start]])
            state[name] = rolled.repeat((n + block.numel() - 1) // block.numel())[:n].view(shape).clone()
    return state, cfg      # fp32 resident, as the reference's own fp32 CPU run would be


def cpu_reference_sample(cfg_full, layers_cpu: int, n_decode: int, threads: int, built=None, repeats: int = 3):
    """One bounded sample of the bench workload on the host: encoders + splice, S-token prefill, `n_decode` greedy
    steps; each phase is the best of `repeats` runs (perf_counter), the layer stack extrapolated x(32 / layers_cpu)."""
    from oracle import vita_oracle as O
    torch.set_num_threads(threads)
    state, cfg = built if built is not None else cpu_reference_state(layers_cpu)
    ids, images, feats, lengths = make_inputs(cfg, pin=False)
    audios = {"audios": feats, "lengths": lengths}
    best = lambda xs: min(xs)
    t_enc, t_prefill, t_dec, t_head = [], [], [], []
    for _ in range(repeats):
        t0 = time.perf_counter()
        img_f = O.encode_images(state, cfg, images)
        aud_f = O.encode_audios(state, cfg, feats, lengths)["inputs_embeds"]
        emb, lens = O.prepare_inputs_embeds(state, cfg, ids, images, audios, img_f, aud_f)
        t_enc.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        logits, past, _ = O.mixtral_forward(state, cfg.llm, emb, last_only=True)
        t_prefill.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for _ in range(n_decode):
            nxt = logits[0, -1].argmax().view(1, 1)
            logits, past, _ = O.forward(state, cfg, nxt, past=past, last_only=True)
        t_dec.append((time.perf_counter() - t0) / max(n_decode, 1))
        # lm_head / embedding cost is inside both measurements once; the layer stack scales with depth
        t0 = time.perf_counter()
        O.linear(torch.zeros(1, cfg.llm.hidden_size), state["lm_head.weight"])
        t_head.append(time.perf_counter() - t0)
    t_enc, t_prefill, t_dec, t_head = best(t_enc), best(t_prefill), best(t_dec), best(t_head)
    scale = cfg_full.llm.num_hidden_layers / layers_cpu
    return dict(S=lens[0], repeats=repeats, t_enc=t_enc, t_prefill=t_prefill, t_dec=t_dec, t_head=t_head,
                t_prefill_full=(t_prefill - t_head) * scale + t_head, t_dec_full=(t_dec - t_head) * scale + t_head)


def pick_cpu_threads() -> int:
    """Fixed rule (recorded in the JSON line): 16 threads, or all of them on a smaller host.  The oracle is plain
    torch on CPU and this workload is many small ops; on the 128-thread GPU box all threads are ~10x slower than 8-16
    (round 1 measured 31 s vs 2.5 s for the encoders), and probing per run made the baseline swing by +-40 %."""
    return min(16, os.cpu_count() or 1)


def cpu_tokens_per_s(sample, new_tokens):
    total = sample["t_enc"] + sample["t_prefill_full"] + new_tokens * sample["t_dec_full"]
    return new_tokens / total


def run_reference(args):
    """--impl reference: the reference algorithm (oracle port) on the host cores.  Every step is its own bounded
    sample of the workload (encoders + S-token prefill + a few decode steps at reduced depth, best of 2 inside the
    sample); the weights are built once."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = VitaConfig.full(args.layers)
    threads = pick_cpu_threads()
    t_all0 = time.perf_counter()
    built = cpu_reference_state(args.cpu_layers)
    t_build = time.perf_counter() - t_all0
    vals, s = [], None
    for i in range(args.warmup + args.steps):
        s = cpu_reference_sample(cfg, args.cpu_layers, args.cpu_decode_tokens, threads, built=built, repeats=2)
        if i >= args.warmup:
            vals.append(cpu_tokens_per_s(s, args.new_tokens))
    v = sum(vals) / len(vals)
    sample = (f"oracle port (fp32, torch CPU, {threads} of {os.cpu_count()} host threads, fixed rule): full "
              f"InternViT+Whale+projector, Mixtral full width x {args.cpu_layers} layer(s), S={s['S']} prompt, "
              f"{args.cpu_decode_tokens} decode steps, every step re-measured (best of 2 per phase); layer stack "
              f"extrapolated x{cfg.llm.num_hidden_layers // args.cpu_layers}: enc {s['t_enc']:.2f}s, prefill "
              f"{s['t_prefill_full']:.2f}s, decode {s['t_dec_full'] * 1e3:.1f} ms/token; min/max over steps "
              f"{min(vals):.3f}/{max(vals):.3f} tokens/s; weights built in {t_build:.0f}s")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * args.new_tokens / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, args, 1),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_all0}
    print(json.dumps(line))


def workload_config(cfg, args, n):
    return {"workload": "configs[2]: 1 image (448x448, 1 tile) + 10 s audio (998 fbank frames) + 126 text tokens -> "
                        f"S={spliced_len(cfg)} omni prefill -> {args.new_tokens}-token greedy decode, bs=1 per GPU",
            "geometry": f"Mixtral-8x7B ({cfg.llm.num_hidden_layers} layers, H=4096, I=14336, 8 experts top-2, "
                        "V=51760) + InternViT-300M + Whale, random init",
            "parallelism": f"replica x{n} (request parallel; the model fits one 180 GB B200)",
            "l2_policy": "inputs larger than L2 (93.7 GB of weights streamed every step)"}


def dump_outputs(out_dir, arrays):
    """Writes each tensor as <out_dir>/<name>.npy (float32, or float64 as given), so that two builds run with the same
    arguments, and hence the same seeded weights and inputs, can be compared output for output."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        assert t.dtype in (torch.float32, torch.float64), name
        np.save(d / f"{name}.npy", t.detach().cpu().numpy())


# ================================================================================================ expert-parallel record
def ep_inputs(cfg, S_target=4096, n_frames=8):
    """BASELINE configs[3]: 8 video frames (448 x 448) + 10 s audio + text filling the sequence to S = 4096."""
    g = torch.Generator().manual_seed(4242)
    t2 = cfg.audio.frames_after_subsampling(AUDIO_FRAMES)
    n_text = S_target - n_frames * cfg.vision.out_tokens - cfg.audio.tokens_after_adapter(t2)
    ids = torch.randint(0, cfg.llm.vocab_size, (1, n_text + n_frames + 1), generator=g)
    ids[0, 1:1 + n_frames] = IMAGE_TOKEN_INDEX
    ids[0, 1 + n_frames] = AUDIO_TOKEN_INDEX
    images = torch.randn(n_frames, 3, cfg.vision.image_size, cfg.vision.image_size, generator=g)
    feats = torch.randn(1, AUDIO_FRAMES, cfg.audio.input_dim, generator=g)
    return ids, images, feats, torch.tensor([AUDIO_FRAMES])


def run_ep_record(args, cfg, single_model, dev, rank, world):
    """N > 1: BASELINE configs[3] end to end under expert parallelism -- the video frames through InternViT data-parallel
    over the ranks (+ one NCCL all-gather of the visual tokens), the audio encoder, the splice, and the S = 4096 Mixtral
    prefill with experts and tokens sharded over the N GPUs (MixtralDecoder._prefill_ep_seq).  Rank 0 also runs the same
    input through its single-GPU replica (identical weights: seed 0) for the strong-scaling reference and the
    bit-equality check of the last-row logits."""
    import torch.distributed as dist
    from vita_b200 import weights as W
    from vita_b200.model.vita_mixtral import VITAMixtralForCausalLM
    from vita_b200.parallel import token_range
    S_T, NF = 4096, 8
    ids, images_h, feats_h, lengths = ep_inputs(cfg, S_T, NF)
    packed = W.random_packed(cfg, dev, seed=0, ep=(rank, world))
    model = VITAMixtralForCausalLM(cfg, packed, dev, max_batch=1, max_seq_len=S_T + 64, max_new_tokens=8)
    llm = model.llm
    images_d, feats_d = images_h.to(dev), feats_h.to(dev)
    mine = list(range(rank, NF, world))                         # frames of this rank
    per = (NF + world - 1) // world
    H = cfg.llm.hidden_size
    ev = lambda: torch.cuda.Event(enable_timing=True)
    ids_list = ids.tolist()

    def step():
        e = [ev() for _ in range(5)]
        e[0].record()
        local = torch.zeros(per, cfg.vision.out_tokens, H, dtype=torch.bfloat16, device=dev)
        if mine:
            local[: len(mine)] = model.encode_images(images_d[mine])
        gathered = torch.empty(world, per, cfg.vision.out_tokens, H, dtype=torch.bfloat16, device=dev)
        dist.all_gather_into_tensor(gathered, local)            # frame f sits at [f % world, f // world]
        img_f = gathered.transpose(0, 1).reshape(per * world, cfg.vision.out_tokens, H)[:NF].contiguous()
        e[1].record()
        aud_f = model.encode_audios(feats_d, lengths)["inputs_embeds"]
        e[2].record()
        emb, plan = model.splice_features(ids_list, img_f, aud_f)
        e[3].record()
        llm.reset()
        llm.prefill(emb[0, : plan.lengths[0]].contiguous(), slot=0, want_last_logits=True)
        e[4].record()
        return e, plan.lengths[0]

    for _ in range(2):
        step()
    dist.barrier(); torch.cuda.synchronize()
    n_rep = 3
    a, b = ev(), ev()
    a.record()
    marks = [step() for _ in range(n_rep)]
    b.record()
    torch.cuda.synchronize()
    dist.barrier()
    S = marks[0][1]
    t = torch.tensor([a.elapsed_time(b) / n_rep] + [sum(m[0][i].elapsed_time(m[0][i + 1]) for m in marks) / n_rep
                                                    for i in range(4)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, vit_ms, aud_ms, spl_ms, pre_ms = t.tolist()
    # last-row logits of the EP run: held by the owner of the last token
    owner = next(r for r in range(world) if token_range(S, r, world)[0] <= S - 1 < token_range(S, r, world)[1])
    last = llm.d_logits[:1].clone() if rank == owner else torch.empty(1, cfg.llm.vocab_size, dtype=torch.bfloat16, device=dev)
    dist.broadcast(last, owner)
    rec = None
    if rank == 0:
        # single-GPU reference on the replica of rank 0 (weights seed 0 = the EP model's)
        sl = single_model.llm
        def single():
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            emb1, lens1 = single_model._embeds_for(ids, images_d, {"audios": feats_d, "lengths": lengths})
            e1.record()
            sl.reset()
            sl.prefill(emb1[0, : lens1[0]].contiguous(), slot=0, want_last_logits=True)
            e2.record()
            return e0, e1, e2
        single(); torch.cuda.synchronize()
        one = [single() for _ in range(2)]
        torch.cuda.synchronize()
        one_total = sum(x[0].elapsed_time(x[2]) for x in one) / len(one)
        one_pre = sum(x[1].elapsed_time(x[2]) for x in one) / len(one)
        ref_last = sl.d_logits[:1].clone()
        sl.reset()
        flops = prefill_flops(S, cfg)
        nvl = {"kv_all_gather": S * 2 * cfg.llm.num_key_value_heads * cfg.llm.head_dim * 2 * (world - 1),
               "routed_rows_all_gather": S * (H * 2 + 16) * (world - 1),
               "combine_push_expected": int(2 * S * H * 2 * (world - 1) / world)}
        rec = {"workload": f"configs[3]: {NF} frames 448x448 + 10 s audio + text -> S={S}, expert-parallel prefill",
               "mode": llm.ep_mode, "n_gpus": world, "ms": total_ms,
               "phases_ms": {"vit_frames_data_parallel_plus_all_gather": vit_ms, "audio_encoder": aud_ms,
                             "splice": spl_ms, "mixtral_prefill_ep": pre_ms},
               "prefill_tflops_aggregate": flops / (pre_ms / 1e3) / 1e12,
               "single_gpu_ms": one_total, "single_gpu_prefill_ms": one_pre,
               "speedup_end_to_end": one_total / total_ms, "speedup_prefill": one_pre / pre_ms,
               "strong_scaling_efficiency_prefill": one_pre / pre_ms / world,
               "bit_identical_last_row_logits_vs_single_gpu": bool(torch.equal(last, ref_last)),
               "max_abs_logit_diff": float((last.float() - ref_last.float()).abs().max()),
               "nvlink_bytes_per_layer_all_ranks": nvl,
               "timing": "CUDA events per rank, max over ranks, mean of 3 after 2 warm-ups; barrier + sync both sides"}
    del model, packed
    torch.cuda.empty_cache()
    return rec



# ================================================================================================ GPU arm
def run_b200(args):
    import torch.distributed as dist
    from vita_b200 import ops, weights as W
    from vita_b200.model.vita_mixtral import VITAMixtralForCausalLM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = VitaConfig.full(args.layers)
    NT = args.new_tokens
    packed = W.random_packed(cfg, dev, seed=rank)
    S_LONG = 4096   # BASELINE configs[3] sequence length: single-GPU prefill-only measurement (tensor-core roofline)
    model = VITAMixtralForCausalLM(cfg, packed, dev, max_batch=1,
                                   max_seq_len=max(spliced_len(cfg) + NT + 64,
                                                   0 if (args.no_long_prefill and (world == 1 or args.no_ep)) else S_LONG + 64),
                                   max_new_tokens=NT + 16)
    ids, images_h, feats_h, lengths = make_inputs(cfg, seed=rank)
    images_d, feats_d = images_h.to(dev), feats_h.to(dev)
    S = spliced_len(cfg)
    llm = model.llm

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    last = {}           # the latest step's prefill output, kept by reference for --dump-outputs

    def device_step():
        e = [ev() for _ in range(4)]
        e[0].record()
        emb, lens = model._embeds_for(ids, images_d, {"audios": feats_d, "lengths": lengths})
        e[1].record()
        llm.reset()
        x = emb[0, : lens[0]].contiguous()
        llm.prefill(x, slot=0)          # x is the residual stream: it ends as the last layer's hidden states
        last["prefill_hidden"] = x
        e[2].record()
        for _ in range(NT):
            llm.decode_step(1, use_graph=True)
        e[3].record()
        return e, lens[0]

    never = [lambda output_ids, scores, **kw: bool(output_ids[0, -1] == -1)]   # a criterion that looks at every token

    def e2e_step():
        """The reference demo's call (video_audio_demo.py:257-270): CUDA input_ids / images / audios made from pinned
        HOST tensors inside the timed region, output_scores + return_dict_in_generate + stopping criteria, default
        read-back cadence; the result (token ids) is read back to the host."""
        out = model.generate(ids.to(dev, non_blocking=True), images=images_h.to(dev, non_blocking=True),
                             audios={"audios": feats_h.to(dev, non_blocking=True), "lengths": lengths}, do_sample=False,
                             temperature=0.01, top_p=None, num_beams=1, output_scores=True,
                             return_dict_in_generate=True, max_new_tokens=NT, use_cache=True, stopping_criteria=never)
        return out.sequences.cpu()

    for _ in range(max(args.warmup, 3)):
        device_step()
        torch.cuda.synchronize()
    e2e_step()
    e2e_step()      # second call: the logits-logging decode graph is captured by now

    # ---- timed region: K device-resident steps --------------------------------------------------------------
    barrier()
    ops.launch_count(reset=True)
    if model._captured is not None:
        model._captured.replayed_launches = 0
    with ClockSampler(local) as clk:
        t_all = [ev(), ev()]
        t_all[0].record()
        marks = [device_step() for _ in range(args.steps)]
        t_all[1].record()
        torch.cuda.synchronize()
    barrier()
    eager_launches = ops.launch_count(reset=True)
    total_ms = t_all[0].elapsed_time(t_all[1])
    enc_ms = sum(m[0][0].elapsed_time(m[0][1]) for m in marks) / args.steps
    pre_ms = sum(m[0][1].elapsed_time(m[0][2]) for m in marks) / args.steps
    dec_ms = sum(m[0][2].elapsed_time(m[0][3]) for m in marks) / args.steps
    assert marks[0][1] == S
    enc_replayed = model._captured.replayed_launches if model._captured is not None else 0
    launches = eager_launches + args.steps * NT * llm.launches_per_decode_step + enc_replayed
    toks = llm.generated_tokens(0)
    assert len(toks) == NT and all(0 <= t < cfg.llm.vocab_size for t in toks)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {
            "generated_ids": torch.tensor(toks, dtype=torch.float64),
            "prefill_hidden": last["prefill_hidden"].float(),          # [S, H]: every prompt position, last layer
            "decode_hidden": llm.d_h[0].float(),                       # [H]: last decode step, last layer
        })

    # ---- e2e: the public generate() with HOST inputs (pinned), H2D + D2H inside the timed region ------------
    barrier()
    t0 = [ev(), ev()]
    t0[0].record()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        out = e2e_step()
    t0[1].record()
    torch.cuda.synchronize()
    e2e_wall = time.perf_counter() - w0
    e2e_ms = max(t0[0].elapsed_time(t0[1]), e2e_wall * 1e3) / args.steps
    assert out.shape[1] == TEXT_TOKENS + NT and not out.is_cuda
    e2e_launches = ops.launch_count(reset=True) + args.steps * NT * llm.launches_per_decode_step_with_scores()
    barrier()

    # ---- parity of THIS configuration at full depth (outside every timed region) ----------------------------
    parity = None
    if not args.no_parity and rank == 0:
        try:
            from tests.full_depth import check_mixtral       # the fp32 oracle, layer-streamed on this GPU (checker)
            emb_p, lens_p = model._embeds_for(ids, images_d, {"audios": feats_d, "lengths": lengths})
            parity = check_mixtral(model, emb_p[0, : lens_p[0]].contiguous(), n_tokens=8)
            parity["what"] = (f"{cfg.llm.num_hidden_layers}-layer Mixtral of this workload (S={lens_p[0]} spliced prompt from "
                              "the CUDA encoders) vs the fp32 oracle run layer-streamed on the same GPU (torch fp32, TF32 "
                              "off): last-row logits of the prefill + 8 free-running greedy ids; full-size encoders + "
                              "splice vs the oracle: tests/test_full_depth_gpu.py")
        except Exception as e:   # the measurement stands on its own; report why the check did not run
            parity = {"error": f"{type(e).__name__}: {e}"[:300]}
        llm.reset()
    barrier()

    # ---- long prefill (S = 4096): where the expert GEMMs are compute-bound -----------------------------------
    long_ms = None
    if not args.no_long_prefill:
        emb_long = (torch.randn(S_LONG, cfg.llm.hidden_size, device=dev) * 0.05).to(torch.bfloat16)
        for _ in range(2):
            llm.reset(); llm.prefill(emb_long.clone(), slot=0)
        torch.cuda.synchronize()
        a, b = ev(), ev()
        tot = 0.0
        for _ in range(3):
            llm.reset()
            x = emb_long.clone()
            a.record(); llm.prefill(x, slot=0); b.record(); b.synchronize()
            tot += a.elapsed_time(b)
        long_ms = tot / 3
        llm.reset()

    # ---- dominant kernel ------------------------------------------------------------------------------------
    c = cfg.llm
    # the expert gate/up GEMV (60% of the decode bytes), timed with CUDA events on the launching stream in an eager
    # pass right after the timed region (inside it the step is one CUDA graph)
    lw = packed["llm"]["layers"]

    def launch_all():
        for li in range(len(lw)):
            ops.decode_tc_moe_gate_up(llm.d_h[:1], lw[li]["ln2"], lw[li]["gate"], lw[li]["w13"], llm.d_ids[:1],
                                      llm.d_w[:1], llm.d_act[:1], llm.tc_ws, c.rms_norm_eps)

    # one launch per layer (32 different 470 MB weight sets, far larger than L2), back to back on the stream;
    # average duration = elapsed / launches
    launch_all()
    torch.cuda.synchronize()
    reps, gu_ms = 3, 0.0
    for r in range(reps):
        a, b = ev(), ev()
        a.record()
        launch_all()
        b.record()
        b.synchronize()
        gu_ms += a.elapsed_time(b)
    gu_ms /= reps * len(lw)
    gu_bytes = c.num_experts_per_tok * 2 * c.intermediate_size * c.hidden_size * 2 + c.hidden_size * 2 \
        + c.num_experts_per_tok * c.intermediate_size * 2 + c.num_local_experts * c.hidden_size * 2
    roof_kernel = "tc_gemv_kernel<TcGateUpOp> (decode: fused RMSNorm + router + the 2 selected experts' gate/up rows + SiLU*up)"
    roof_note = ("one launch per layer back to back on the stream, CUDA events around the batch, right after the timed "
                 "region (inside it the decode step is a single CUDA graph)")
    pk = peaks()

    # ---- reduce over ranks (max time) -----------------------------------------------------------------------
    def rmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    total_ms, enc_ms, pre_ms, dec_ms, e2e_ms = map(rmax, (total_ms, enc_ms, pre_ms, dec_ms, e2e_ms))
    step_ms = total_ms / args.steps
    if rank == 0:
        ctx_mid = S + NT // 2
        dec_tok_s = NT / (dec_ms / 1e3)
        line = {
            "metric": METRIC, "value": world * NT / (step_ms / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(cfg, args, world),
            "phases_ms": {"encoders_and_splice": enc_ms, "mixtral_prefill": pre_ms, "decode_total": dec_ms,
                          "decode_per_token": dec_ms / NT},
            "decode": {"tokens_per_s_per_gpu": dec_tok_s, "algorithmic_gb_per_token": decode_bytes(ctx_mid, cfg) / 1e9,
                       "hbm_gbs": decode_bytes(ctx_mid, cfg) / 1e9 * dec_tok_s, "hbm_frac": decode_bytes(ctx_mid, cfg)
                       / 1e9 * dec_tok_s / pk["hbm_gbs"]},
            "prefill": {"S": S, "tflops": prefill_flops(S, cfg) / (pre_ms / 1e3) / 1e12,
                        "tensor_frac": prefill_flops(S, cfg) / (pre_ms / 1e3) / 1e12 / pk["tflops"],
                        "encoders_tflops": encoder_flops(cfg) / (enc_ms / 1e3) / 1e12},
            "roofline": {"kernel": roof_kernel, "how": roof_note, "bound": "hbm", "achieved": gu_bytes / 1e9 / (gu_ms / 1e3),
                         "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gu_bytes / 1e9 / (gu_ms / 1e3) / pk["hbm_gbs"],
                         "traffic": ncu_traffic_bytes(roof_kernel), "bytes_per_launch": gu_bytes,
                         "us_per_launch": gu_ms * 1e3, "peak_source": pk["source"],
                         "traffic_source": "profiles/r02_prof_tc_gateup_full.md (ncu --set full, one launch, "
                                           "dram__bytes_read.sum + dram__bytes_write.sum)"},
            "prefill_long": None if long_ms is None else {
                "S": S_LONG, "ms": long_ms, "tflops": prefill_flops(S_LONG, cfg) / (long_ms / 1e3) / 1e12,
                "tensor_frac": prefill_flops(S_LONG, cfg) / (long_ms / 1e3) / 1e12 / pk["tflops"],
                "note": "Mixtral prefill only, 32 layers, one GPU, random embeddings (BASELINE configs[3] length)"},
            "e2e": {"value": world * NT / (e2e_ms / 1e3), "unit": UNIT,
                    "h2d_bytes_per_step": images_h.numel() * 4 + feats_h.numel() * 4 + ids.numel() * 8,
                    "d2h_bytes_per_step": NT * 4 + (TEXT_TOKENS + NT) * 8, "ms_per_step": e2e_ms,
                    "call": "model.generate(input_ids.cuda(), images=..., audios=..., do_sample=False, output_scores=True, "
                            "return_dict_in_generate=True, max_new_tokens=256, use_cache=True, stopping_criteria=[...]) "
                            "as video_audio_demo.py:257-270; CUDA-graph decode with the device-side logits log",
                    "gpu_launches": int(e2e_launches)},
            "parity": parity,
            "ep": None,
            "gpu_launches": int(launches),
            "clocks": clk.summary(),
        }
        if world == 1 and not args.no_cpu_baseline:
            threads = pick_cpu_threads()
            s = cpu_reference_sample(cfg, args.cpu_layers, args.cpu_decode_tokens, threads, repeats=3)
            line["cpu_baseline"] = {
                "value": cpu_tokens_per_s(s, NT), "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"oracle port fp32, {threads} of {os.cpu_count()} host threads (fixed rule): encoders full "
                          f"size, Mixtral full width x{args.cpu_layers} layer(s) (stack extrapolated to "
                          f"{cfg.llm.num_hidden_layers}), S={s['S']}, {args.cpu_decode_tokens} decode steps, best of 3 "
                          f"per phase: enc {s['t_enc']:.2f}s prefill {s['t_prefill_full']:.2f}s decode "
                          f"{s['t_dec_full'] * 1e3:.1f} ms/token"}
    else:
        line = None

    # ---- N > 1: the expert-parallel configs[3] record, LAST (collective over all ranks).  Everything above is already
    # in `line`; a watchdog prints it without the record if the exchange protocol ever hangs, a Python / CUDA error
    # lands in ep.error -- the replica measurement is never lost to this step.
    if world > 1 and not args.no_ep:
        done = threading.Event()

        def bail():
            if not done.is_set():
                if line is not None:
                    line["ep"] = {"error": "expert-parallel record did not finish within 240 s"}
                    print(json.dumps(line), flush=True)
                os._exit(0)

        timer = threading.Timer(240.0, bail)
        timer.daemon = True
        timer.start()
        try:
            ep_rec = run_ep_record(args, cfg, model, dev, rank, world)
        except Exception as e:
            ep_rec = {"error": f"{type(e).__name__}: {e}"[:400]}
        done.set()
        timer.cancel()
        if line is not None:
            line["ep"] = ep_rec
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


def ncu_traffic_bytes(kernel_name: str):
    """DRAM bytes of one launch of the roofline kernel, from the committed ncu --set full summary (None if the active
    decode path is not the profiled kernel or the summary is missing)."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_prof_tc_gateup_full.md")
    if "TcGateUpOp" not in kernel_name or not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    for ln in open(path):
        c = [x.strip() for x in ln.strip().strip("|").split("|")]
        if len(c) >= 3 and c[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and c[2] in unit:
            tot += float(c[1]) * unit[c[2]]
    return tot or None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--new-tokens", type=int, default=256)
    ap.add_argument("--cpu-layers", type=int, default=2)
    ap.add_argument("--cpu-decode-tokens", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-long-prefill", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-depth fp32-oracle check of the workload")
    ap.add_argument("--no-ep", action="store_true", help="N > 1: skip the expert-parallel configs[3] record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results (rank 0) to DIR/<name>.npy: generated_ids, "
                         "prefill_hidden (the prefill's last-layer hidden states), decode_hidden (the last decode "
                         "step's last-layer hidden state)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
