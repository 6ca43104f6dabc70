#!/usr/bin/env python
"""bench.py -- the vAttention hot path on B200, BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|fa_vattn]
                    [--workload decode32k|tp70b] [--ctx C] [--dump-outputs DIR]

Workload "decode32k" (default; BASELINE.json configs[1]): Llama-3-8B attention shapes (Hq 32,
Hkv 8, D 128, 32 layers, hidden 4096), batch 64, 32K context, K/V in vAttention virtual tensors
with 2 MiB pages (fa_vattn_2mb).  One STEP = one decode iteration of the path: allocator
step_async(seq_lens) + 32 layer-calls of [flash_attn_with_kvcache(q[64,1], K, V, k_new, v_new,
cache_seqlens, cache_batch_idx) (append + attention) -> row-parallel o_proj GEMM (+ all-reduce
for N > 1)], producing 64 tokens.  The 32 layer-calls are replayed from a CUDA graph at every N
(cache_seqlens is a device tensor the graph increments; step_async stays outside).  Sequence
lengths straddle the 32K page boundary -- sequence b crosses it at a different step, the crossings
spread over a fixed fraction (1/46) of the rank's page at every N -- so the timed steps make the
allocator map pages (reported: on the critical path / in the background, the device time of every
timed step, and how many step_async calls were queued behind a mapper pass still in flight).
Full-model KV at this shape is 256 GiB, so (like the reference's own
microbenchmarks/perf_pagesize/bench_pagesize.py:22) only a few layers are resident and the layer
calls rotate over them; each call still streams its own 8.6 GB, far beyond the 126 MB L2.

Workload "tp70b" (configs[4]): Llama-3-70B (Hq 64, Hkv 8, D 128, 80 layers, hidden 8192), batch
16, --ctx 32768 | 65536 | 131072 (scripts/benchmark_e2e_static_trace.py:12,30); meant for
--gpus 8 (Hq 8 / Hkv 1 per GPU), runs at any N that divides 8.

metric  decode tokens/s (attention path) = batch * K / t_K_steps, device-timed, max over ranks.
e2e     the attention call through the host-buffer C-ABI entry point (vattn_fwd_kvcache_host*):
        q/k/v/index arrays start in pinned host memory every call, the output is read back.
roofline  dominant kernel = the decode attention sweep; algorithmic bytes per launch (SURVEY 8d)
        / its average device duration, taken with CUDA events around that kernel over K eager
        iterations right after the timed region (events cannot be read back from inside a
        graph), against the measured HBM copy bandwidth.
parity_check  before timing, one layer-call at the timed shape is compared with
        flash_attn.flash_attn_with_kvcache on identical inputs (1e-3 * scale + 1 output ulp; the
        appended rows bit-identical) and, on sampled rows, with an fp32 torch reference; for
        N > 1 the fused o_proj + all-reduce output is compared with the fp32 sum of the ranks'
        16-bit partials and must be bit-identical on every rank.  A failure raises.
extras (N == 1, decode32k)  short legs for the other figures BASELINE's metric names:
        "prefill" (configs[2]: Yi-6B 128K chunked prefill TFLOP/s), "pod" (configs[3]: 8x16K
        prefill + 56x4K decode, and the balanced hybrid batch the POD wrapper issues; serial vs
        fused), "fa_vattn" (the reference's GPU dispatch target, flash_attn over the same
        virtual tensors / shapes, on the same box).
N > 1   head-sharded tensor parallel (SURVEY 8e): rank r owns Hq/N q heads and Hkv/N kv heads and
        its own allocator; per layer-call ONE all-reduce sums the [batch, hidden] o_proj partials
        -- by default inside our fused GEMM + all-reduce kernel (--tp-collective fused|peer|nccl).
        The model is fixed, so per-GPU work shrinks with N: "scaling": "strong" (at every N).
--impl reference   the reference's CPU path for the same metric: torch SDPA over the same shapes
        on the host cores (oracle/attention_ref.sdpa_decode_cpu), a bounded sample per step.
--impl fa_vattn    the reference's own GPU path on this box: its vattention extension compiled
        unmodified (oracle/_ref) allocates the virtual tensors, flash_attn attends over them.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from dataclasses import dataclass
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

PAGE = 2 << 20
DTYPE = torch.bfloat16
D = 128


@dataclass(frozen=True)
class Workload:
    name: str
    hq: int
    hkv: int
    layers: int
    hidden: int
    batch: int
    ctx: int
    model: str


def workload_from(args) -> Workload:
    if args.workload == "tp70b":
        # Llama-3-70B (pod_attn/tests/utils.py, scripts/benchmark_e2e_static_trace.py:12,30)
        return Workload("tp70b", 64, 8, 80, 8192, 16, args.ctx or 32768, "Llama-3-70B")
    return Workload("decode32k", 32, 8, 32, 4096, 64, args.ctx or 32768, "Llama-3-8B")


def rank_info():
    return (int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)),
            int(os.environ.get("WORLD_SIZE", 1)))


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            d = json.loads(f.read_text())
            return (float(d["hbm_gbs"]), float(d["bf16_tflops"]), float(d["bf16_tflops_sustained"]),
                    "measured (MEASURED_PEAKS.json)")
        except Exception:
            pass
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(gpu_index), "-lms", "100"], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [l.strip().split(", ") for l in open(self.tmp.name) if l.strip()]
        os.unlink(self.tmp.name)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.strip().lower() == "active":
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "samples": len(sm),
                "reasons": sorted(reasons)}


def algorithmic_bytes(total_len_after_append: float, hq, hkv, batch) -> int:
    """SURVEY 8(d): K and V read once (incl. the appended token) + Q read / O write + k/v new write."""
    itemsize = 2
    return int(2 * itemsize * hkv * D * total_len_after_append
               + 2 * itemsize * batch * hq * D + 2 * itemsize * batch * hkv * D)


ULP = {torch.bfloat16: 2.0 ** -7, torch.float16: 2.0 ** -10}


def close_to_library(ours, lib):
    """bf16 criterion of tests/test_gpu_baseline_configs.py: rms(ours - lib) <= 1e-3 * max|lib| and
    |ours - lib| <= 8e-3 * max|lib| + one output ulp of |lib_i| (two implementations that both round
    P to bf16, as FA-2 does, differ by that much at 32K keys)  ->  (ok, max_diff / scale, rms / scale)."""
    a, b = ours.float(), lib.float()
    scale = max(b.abs().max().item(), 1e-30)
    err = (a - b).abs()
    bad = int((err > 8e-3 * scale + ULP[ours.dtype] * b.abs()).sum().item())
    rms = float((err.double() ** 2).mean().sqrt().item())
    ok = bad == 0 and rms <= 1e-3 * scale and not bool(torch.isnan(a).any())
    return ok, err.max().item() / scale, rms / scale


def fp32_decode_rows(q, kc, vc, lens_after, slots, rows, scale):
    """fp32 torch reference of decode attention for a few batch rows (the appended token already in
    the cache): q [B,1,Hq,D], caches [slots,S,Hkv,D] -> [len(rows),1,Hq,D]."""
    out = []
    g = q.shape[2] // kc.shape[2]
    for b in rows:
        n = int(lens_after[b])
        k = kc[int(slots[b]), :n].float().repeat_interleave(g, dim=1)        # [n, Hq, D]
        v = vc[int(slots[b]), :n].float().repeat_interleave(g, dim=1)
        s = torch.einsum("hd,nhd->hn", q[b, 0].float(), k) * scale
        p = torch.softmax(s, dim=-1)
        out.append(torch.einsum("hn,nhd->hd", p, v))
    return torch.stack(out).unsqueeze(1)


# ------------------------------------------------------------------------------- ours ---

def crossing_schedule(batch: int, ctx: int, tpp: int, tpp_unsharded: int, warmup: int, steps: int, total_steps: int):
    """Start lengths that make sequences cross the page boundary at `ctx` one after another during the run.

    Sequence b starts off_b + 1 tokens below the boundary (plus the untimed steps before the timed
    region), off_b spread evenly over `spread` tokens.  `spread` is a fixed FRACTION of this rank's page
    (tokens per page grow with N as the kv heads are sharded): page crossings come ~45x more often
    than with uniformly distributed lengths at every N -- the same token stream maps the same BYTES
    per step on every rank count, not N times more.  Returns (spread, lengths)."""
    spread = max(8, min(total_steps, 2 * (warmup + steps))) * (tpp // tpp_unsharded)
    return spread, [ctx - (b * spread) // batch - 1 - (warmup + 2) for b in range(batch)]


def run_ours(args):
    wl = workload_from(args)
    rank, local_rank, world = rank_info()
    assert world == args.gpus, f"WORLD_SIZE {world} != --gpus {args.gpus}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from vattention_b200 import attention as att
    from vattention_b200 import vattention as va
    from vattention_b200.tp import (HeadShard, HeadShardedAttention, HeadShardedAttentionFused,
                                    HeadShardedAttentionPeer)

    shard = HeadShard(rank, world, wl.hq, wl.hkv, D)
    hq, hkv = shard.heads_per_rank, shard.kv_heads_per_rank
    B, LAYERS, HIDDEN, CTX = wl.batch, wl.layers, wl.hidden, wl.ctx
    K, W = args.steps, args.warmup
    tpp = PAGE // (hkv * D * 2)                     # tokens per 2 MiB page of this rank's shard
    assert CTX % tpp == 0, "the context must end on a page boundary for the crossing schedule"
    # every step of the run, in order: graph warm-up (2) + W + K timed + K eager (kernel timing) +
    # e2e (W + K) + parity (1)
    total_steps = 3 + W + K + K + (0 if args.no_e2e else W + K) + 2
    spread, seq_lens = crossing_schedule(B, CTX, tpp, PAGE // (wl.hkv * D * 2), W, K, total_steps)
    torch.zeros(1, device=dev)                  # context for the allocator (cudaInternal.h:19-25)
    n_res = args.resident_layers
    max_ctx = CTX + tpp                          # one page of head-room past the boundary
    tensors = va.init_kvcache(n_res, hkv, D, B, max_ctx, local_rank, DTYPE, PAGE, False)
    per_layer_bytes = 2 * B * max_ctx * hkv * D * 2
    va.reserve_physical_pages(n_res * per_layer_bytes)
    va.set_compute_stream(torch.cuda.current_stream(dev).cuda_stream, True)
    k_layers, v_layers = tensors[:n_res], tensors[n_res:]
    # the serving loop's slot assignment: alloc_new_batch_idx per sequence, then a shuffled
    # cache_batch_idx like the reference's microbenchmarks
    rids = [va.alloc_new_batch_idx(seq_lens[i]) for i in range(B)]
    assert sorted(rids) == list(range(B))
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0))
    slot_of = perm.tolist()                       # request b lives in cache slot perm[b]
    slot_lens = [0] * B                           # the allocator's view: lengths per slot (reqId)
    for b in range(B):
        slot_lens[slot_of[b]] = seq_lens[b]
    va.step_async(slot_lens)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    for t in list(k_layers) + list(v_layers):
        for s in range(B):
            t[s, :slot_lens[s]].normal_(generator=g)
    batch_idx = perm.int().to(dev)
    q = torch.randn(LAYERS, B, 1, hq, D, device=dev, generator=g).to(DTYPE)
    kn = torch.randn(LAYERS, B, 1, hkv, D, device=dev, generator=g).to(DTYPE)
    vn = torch.randn(LAYERS, B, 1, hkv, D, device=dev, generator=g).to(DTYPE)
    # row-parallel o_proj shard [Hq/N * D, hidden] (tensor_parallel/layers.py:432-447)
    w_o = (torch.randn(hq * D, HIDDEN, device=dev, generator=g) * 0.02).to(DTYPE)
    scale = D ** -0.5
    sink = torch.zeros(1, device=dev, dtype=torch.float32)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- the o_proj GEMM (+ all-reduce) arrangement ------------------------------------------
    tp_attn = None
    if world > 1:
        def all_ranks_ok(ok: bool) -> bool:
            t = torch.tensor([0 if ok else 1], device=dev, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return int(t.item()) == 0

        if args.tp_collective == "fused":
            # our GEMM + all-reduce kernel; probed once (symmetric-memory rendezvous, one exchange) and
            # replaced by the cuBLAS + NCCL pair on EVERY rank if any rank could not bring it up
            ok = True
            try:
                tp_attn = HeadShardedAttentionFused(shard, w_o, att.flash_attn_with_kvcache, max_tokens=B)
                tp_attn.op(torch.zeros(B, hq * D, device=dev, dtype=DTYPE))
                torch.cuda.synchronize(dev)
                ok = not tp_attn.op.failed()
            except Exception as e:                       # noqa: BLE001 -- any failure means "fall back"
                print(f"[bench] rank {rank}: fused o_proj + all-reduce unavailable: {e}", file=sys.stderr)
                ok = False
            if not all_ranks_ok(ok):
                args.tp_collective = "nccl"
        if args.tp_collective == "peer":
            tp_attn = HeadShardedAttentionPeer(shard, w_o, att.flash_attn_with_kvcache, max_tokens=B)
        elif args.tp_collective == "nccl":
            tp_attn = HeadShardedAttention(shard, w_o, att.flash_attn_with_kvcache)
    else:
        # one GPU: no collective, the o_proj is a plain library GEMM (cuBLAS) after the attention call
        tp_attn = HeadShardedAttention(shard, w_o, att.flash_attn_with_kvcache)

    cs = torch.tensor(seq_lens, dtype=torch.int32, device=dev)   # cached length per REQUEST (device)

    def advance(lens_now):
        """Host side of one decode iteration: lengths after this step's token, pages mapped."""
        new = [n + 1 for n in lens_now]
        for b in range(B):
            slot_lens[slot_of[b]] = new[b]
        va.step_async(slot_lens)                  # pages for this token are mapped on return
        return new

    # graph replays need static shapes: the views end at a bound no sequence reaches during the run
    # (the wrapper's per-step slice [:, :max_cache_len], vattention_flashattention_wrapper.py:197, with
    # the maximum taken over the whole run)
    static_len = min(max_ctx, max(seq_lens) + total_steps + 8)
    step_out = [None] * LAYERS                   # the latest step's layer-call outputs (--dump-outputs)

    def layers_body(full_views: bool, max_len: int = 0):
        for layer in range(LAYERS):
            kc, vc = k_layers[layer % n_res], v_layers[layer % n_res]
            kc, vc = (kc[:, :static_len], vc[:, :static_len]) if full_views else (kc[:, :max_len], vc[:, :max_len])
            step_out[layer] = tp_attn.forward(q[layer], kc, vc, kn[layer], vn[layer], cache_seqlens=cs,
                                              cache_batch_idx=batch_idx, softmax_scale=scale, causal=True)
        sink.add_(step_out[-1].flatten()[0].float())
        cs.add_(1)

    def eager_step(lens_now):
        new = advance(lens_now)
        layers_body(False, max(new))
        return new

    # ---- parity check at the timed shape (before any timing) -----------------------------------
    parity = parity_check(att, dist, dev, rank, world, wl, shard, tp_attn, w_o, q[0], kn[0], vn[0],
                          k_layers[0], v_layers[0], cs, batch_idx, seq_lens, slot_of, scale, args)
    barrier()        # (the parity call wrote layer 0's row `len`; the first step writes the same bytes again)

    # ---- CUDA graph of the layer-calls (peer arm: eager, its epoch is a host-side argument) ----
    use_graph = args.graph and args.tp_collective != "peer"
    one_step = eager_step
    graph_launches = 0
    if use_graph:
        seq_lens = advance(seq_lens)              # one eager iteration on a side stream (loads modules,
        side = torch.cuda.Stream(device=dev)      # sizes workspaces for the full-extent views)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            layers_body(True)
        torch.cuda.current_stream(dev).wait_stream(side)
        barrier()
        graph = torch.cuda.CUDAGraph()
        n0 = att.launch_count()
        seq_lens = advance(seq_lens)
        with torch.cuda.graph(graph):
            layers_body(True)
        graph_launches = att.launch_count() - n0
        graph.replay()                            # capture does not execute: run this step for real
        barrier()

        def one_step(lens_now):                   # noqa: F811 -- the graph-replay flavour of one_step
            new = advance(lens_now)
            graph.replay()
            return new

    for _ in range(W):
        seq_lens = one_step(seq_lens)
    barrier()
    launches0 = att.launch_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total_len_first = sum(seq_lens)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    st0 = va.get_step_stats()                     # (waits for the mapper: the warm-up's last pass is done)
    e0.record()
    for i in range(K):
        seq_lens = one_step(seq_lens)             # step_async + graph replay: nothing here waits for the mapper
        marks[i].record()                         # unless this step needs a page it has not mapped yet
    e1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    dumped = None
    if args.dump_outputs and rank == 0:
        # what the last timed step handed back: every layer-call's block output (the fused and peer
        # collectives return one internal buffer, valid until the next call: then only the last
        # layer's survives) and the K/V rows it appended to the resident layers' caches
        outs = step_out if len({t.data_ptr() for t in step_out}) == LAYERS else step_out[-1:]
        pos, slots = (cs - 1).long(), batch_idx.long()
        dumped = {"block_out": torch.stack(outs).cpu(),
                  "k_appended": torch.stack([t[slots, pos] for t in k_layers]).cpu(),
                  "v_appended": torch.stack([t[slots, pos] for t in v_layers]).cpu()}
    ms = e0.elapsed_time(e1)
    step_ms = [round(a.elapsed_time(b), 3) for a, b in zip([e0] + marks[:-1], marks)]
    st1 = va.get_step_stats()                     # totals since init_kvcache; the difference is the timed region
    crit_pages, bg_pages = (st1[k] - st0[k] for k in ("total_sync_pages", "total_async_pages"))
    crit_ns, bg_ns = (st1[k] - st0[k] for k in ("total_critical_path_ns", "total_background_ns"))
    queued_steps = st1["queued_steps"] - st0["queued_steps"]
    launches = (att.launch_count() - launches0) + graph_launches * K if use_graph else att.launch_count() - launches0
    # per-launch time of the dominant kernel: K eager iterations of the same step right after the
    # timed region (events cannot be read back from inside a graph)
    att.kernel_timing(1)
    total_len_eager = sum(seq_lens)
    for _ in range(K):
        seq_lens = eager_step(seq_lens)
    barrier()
    kern_ms, kern_n = att.kernel_timing(2)
    att.kernel_timing(0)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = B * K / (ms / 1e3)

    # roofline of the dominant kernel (per launch = one layer-call on this rank's head shard)
    mean_total_after = total_len_eager + B * (K + 1) / 2.0
    bytes_per_launch = algorithmic_bytes(mean_total_after, hq, hkv, B)
    hbm_peak, _, _, peak_src = peaks()
    roof = None
    if kern_n:
        achieved = bytes_per_launch / (kern_ms / kern_n * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                "frac": round(achieved / hbm_peak, 4),
                "traffic": TRAFFIC_CAPTURE["bytes"] if (world == 1 and wl.name == "decode32k") else None,
                "traffic_source": TRAFFIC_CAPTURE["source"] if (world == 1 and wl.name == "decode32k") else None,
                "kernel_ms_per_launch": round(kern_ms / kern_n, 4), "launches_timed": kern_n,
                "kernel_timed": "K eager iterations after the timed region, CUDA events around the kernel",
                "algorithmic_bytes_per_launch": int(bytes_per_launch), "peak_source": peak_src}

    # ---- e2e: host buffers through the C ABI ------------------------------------------
    e2e = None
    if not args.no_e2e:
        qh = q.cpu().pin_memory()
        knh, vnh = kn.cpu().pin_memory(), vn.cpu().pin_memory()
        idx_h = perm.int().pin_memory()
        outh_l = [torch.empty(B, 1, hq, D, dtype=DTYPE).pin_memory() for _ in range(2)]
        sl_h = torch.empty(B, dtype=torch.int32).pin_memory()
        pin_partial = torch.empty(B, HIDDEN, dtype=DTYPE).pin_memory() if world > 1 else None

        def one_step_e2e(lens_now):
            new = advance(lens_now)
            sl_h.copy_(torch.tensor(lens_now, dtype=torch.int32))
            max_len = max(new)
            part = None
            for layer in range(LAYERS):
                kc = k_layers[layer % n_res][:, :max_len]
                vc = v_layers[layer % n_res][:, :max_len]
                if world == 1:
                    # enqueue only; one stream synchronisation per decode iteration (below) delivers
                    # the result of the last layer to the host
                    att.flash_attn_with_kvcache_host(qh[layer], kc, vc, knh[layer], vnh[layer], sl_h, idx_h,
                                                     outh_l[layer & 1], softmax_scale=scale, causal=True,
                                                     wait=False, pipelined=True)
                else:
                    qd = qh[layer].to(dev, non_blocking=True)
                    knd, vnd = knh[layer].to(dev, non_blocking=True), vnh[layer].to(dev, non_blocking=True)
                    sld, idd = sl_h.to(dev, non_blocking=True), idx_h.to(dev, non_blocking=True)
                    part = tp_attn.forward(qd, kc, vc, knd, vnd, cache_seqlens=sld, cache_batch_idx=idd,
                                           softmax_scale=scale, causal=True)
                    if rank == 0:
                        # the all-reduced block output is replicated: one rank hands it to the host
                        pin_partial.copy_(part, non_blocking=True)
            if world == 1:
                att.host_pipeline_join(dev)
            torch.cuda.current_stream(dev).synchronize()
            return new

        for _ in range(W):
            seq_lens = one_step_e2e(seq_lens)
        barrier()
        e0.record()
        for _ in range(K):
            seq_lens = one_step_e2e(seq_lens)
        e1.record()
        barrier()
        ms_e = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms_e], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e = float(t.item())
        h2d = LAYERS * (B * hq * D * 2 + 2 * B * hkv * D * 2 + 2 * B * 4)
        d2h = LAYERS * (B * (HIDDEN if world > 1 else hq * D) * 2)
        e2e = {"value": round(B * K / (ms_e / 1e3), 2), "unit": "tokens/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": round(ms_e / K, 3),
               "api": ("vattn_fwd_kvcache_host_pipelined per layer-call (copies on their own streams) + join + one "
                       "stream sync per step (C ABI: pinned host q/k/v/idx in, attention output out; no o_proj on "
                       "this boundary; measured 1679 vs 1606 tokens/s for the in-line copies of "
                       "vattn_fwd_kvcache_host_async)") if world == 1
               else "pinned host -> HeadShardedAttention.forward (attention + o_proj + all-reduce) -> pinned host "
                    "on rank 0 (the output is replicated)"}

    if world > 1 and args.tp_collective == "fused" and tp_attn.op.failed():
        raise RuntimeError("fused o_proj + all-reduce: a peer did not arrive (device-side spin limit)")
    cfg_alloc = va.get_config()
    va.cleanup()

    # ---- the other figures of BASELINE's metric + the same-box library comparison (N == 1) ----
    extras = {}
    if world == 1 and wl.name == "decode32k" and not args.no_extras:
        for name, fn in (("prefill", extra_prefill), ("pod", extra_pod), ("fa_vattn", extra_fa_vattn)):
            try:
                extras[name] = fn(att, va, dev, wl)
            except Exception as e:                       # noqa: BLE001 -- a leg must not lose the headline
                extras[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            try:
                va.cleanup()
            except Exception:                            # noqa: BLE001
                pass
            torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, N == 1) ---------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(wl, sample_seqs=args.cpu_sample_seqs, budget_s=args.cpu_budget_s)

    if rank == 0:
        line = {
            "metric": f"decode tokens/s @{CTX // 1024}K ctx ({wl.model} attention path)", "value": round(value, 2),
            "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms / K, 3), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": f"synthetic N(0,1) q/k/v, lengths straddling the {CTX // 1024}K page boundary "
                    f"(mean {total_len_first / B + K / 2:.0f}, crossings spread over {spread} tokens = 1/{tpp // spread} of a "
                    f"page), shuffled cache_batch_idx",
            "config": {"workload": wl.name,
                       "shapes": f"B{B} Hq{wl.hq} Hkv{wl.hkv} D{D} L{LAYERS} ctx{CTX} hidden{HIDDEN}",
                       "backend": "fa_vattn_2mb (vAttention virtual tensors, 2 MiB pages, step_async)",
                       "resident_layers": n_res, "parallelism": f"tp{world}" if world > 1 else "single",
                       "layer_call": "attention (append + decode sweep) + row-parallel o_proj GEMM" +
                                     (" + all-reduce" if world > 1 else ""),
                       "collective": (f"o_proj + all-reduce [{B},{HIDDEN}] bf16 per layer-call: " + {
                           "fused": "ONE kernel: tcgen05 GEMM, tiles exchanged over NVLink peer memory and "
                                    "reduced in place (csrc/oproj_allreduce.cu)",
                           "peer": "cuBLAS GEMM + one-shot all-reduce kernel over NVLink peer memory "
                                   "(csrc/tp_allreduce.cu)",
                           "nccl": "cuBLAS GEMM + NCCL all-reduce"}[args.tp_collective]) if world > 1
                       else "none (one GPU): o_proj is a cuBLAS GEMM",
                       "cuda_graph": bool(use_graph),
                       "l2": f"each layer-call streams {bytes_per_launch / 1e9:.2f} GB of K/V over {n_res} rotating "
                             "layers (>> 126 MB L2); no flush needed" if bytes_per_launch * n_res > (512 << 20)
                             else "working set below 4x L2: see config.resident_layers",
                       "ms_per_layer_call": round(ms / K / LAYERS, 4)},
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
            "clocks": clocks, "parity_check": parity,
            "allocator": {"tokens_per_page": cfg_alloc["tokens_per_page"],
                          "pages_mapped_on_critical_path": int(crit_pages),
                          "pages_mapped_in_background": int(bg_pages),
                          "timed_steps": K, "resident_layers": n_res,
                          "step_async_critical_path_us_mean": round(crit_ns / K / 1e3, 1),
                          "background_pass_us_mean": round(bg_ns / K / 1e3, 1),
                          "background_pass_us_max_since_init": round(st1["max_background_ns"] / 1e3, 1),
                          "steps_queued_behind_a_pass": int(queued_steps),
                          "device_ms_of_each_timed_step": step_ms,
                          "note": "pages of 2 MiB mapped during the K timed steps (K and V, resident layers "
                                  "only); background = the mapper thread under the previous step's kernels"},
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each tensor as <out_dir>/<name>.npy in float32, so that two builds run with the same
    arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np
    total = sum(t.numel() * 4 for t in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().numpy())


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of decode_tc_kernel on the decode32k
# shapes, from an `ncu --set full` capture -- not a measurement of this run (profiles/README.md)
TRAFFIC_CAPTURE = {"bytes": 8610056664,
                   "source": "ncu --set full capture of one launch of this command's decode_tc_kernel, "
                             "profiles/r2_decode_tc_headline_ncu_raw.csv (dram read 8.590103 GB + write "
                             "19.95 MB; 1.002 x algorithmic; lengths straddling the page boundary)"}


def parity_check(att, dist, dev, rank, world, wl, shard, tp_attn, w_o, q0, kn0, vn0, kc, vc, cs, batch_idx,
                 seq_lens, slot_of, scale, args) -> dict:
    """One layer-call at the timed shape against the library / an fp32 reference; raises on failure."""
    B = wl.batch
    res = {"shape": f"B{B} Hq{shard.heads_per_rank} Hkv{shard.kv_heads_per_rank} lens {min(seq_lens)}..{max(seq_lens)}"}
    max_len = max(seq_lens) + 1
    kv, vv = kc[:, :max_len], vc[:, :max_len]
    want = None
    try:
        from flash_attn import flash_attn_with_kvcache as fa
        # same cache: both calls write the same bytes to the same rows before attending
        want = fa(q0, kv, vv, kn0, vn0, cache_seqlens=cs, cache_batch_idx=batch_idx, softmax_scale=scale, causal=True)
        rows_lib = torch.stack([kv[slot_of[b], seq_lens[b]].clone() for b in (0, B // 2, B - 1)])
    except Exception as e:                               # noqa: BLE001 -- library absent / not runnable
        res["flash_attn"] = f"unavailable: {type(e).__name__}"
    out = att.flash_attn_with_kvcache(q0, kv, vv, kn0, vn0, cache_seqlens=cs, cache_batch_idx=batch_idx,
                                      softmax_scale=scale, causal=True)
    torch.cuda.synchronize(dev)
    if want is not None:
        ok, rel, rms = close_to_library(out, want)
        rows_ours = torch.stack([kv[slot_of[b], seq_lens[b]] for b in (0, B // 2, B - 1)])
        res["vs_flash_attn"] = {"ok": ok, "max_diff_over_scale": round(rel, 6), "rms_diff_over_scale": round(rms, 6),
                                "tolerance": "rms <= 1e-3 * max|lib|, max <= 8e-3 * max|lib| + 1 bf16 ulp "
                                             "(bf16 P rounding, see tests/test_gpu_baseline_configs.py)",
                                "appended_rows_bit_identical": bool(torch.equal(rows_ours, rows_lib))}
        if not ok or not torch.equal(rows_ours, rows_lib):
            raise RuntimeError(f"parity_check failed against flash_attn: {res}")
    rows = [0, B // 2, B - 1]
    ref = fp32_decode_rows(q0, kv, vv, [n + 1 for n in seq_lens], slot_of, rows, scale)
    err = (out[rows].float() - ref).abs()
    s = ref.abs().max().item()
    ok32 = bool((err <= 3e-3 * s + ULP[DTYPE] * ref.abs()).all())
    res["vs_fp32_rows"] = {"ok": ok32, "rows": rows, "max_err_over_scale": round(err.max().item() / s, 6),
                           "tolerance": "3e-3 * max|ref| + 1 bf16 ulp (P is rounded to bf16 as in FA-2)"}
    if want is not None:
        e_lib = (want[rows].float() - ref).abs().max().item()
        res["vs_fp32_rows"]["library_max_err_over_scale"] = round(e_lib / s, 6)
        ok32 = ok32 and err.max().item() <= 1.5 * e_lib + ULP[DTYPE] * s
    if not ok32:
        raise RuntimeError(f"parity_check failed against the fp32 reference: {res}")
    if world > 1:
        # fused o_proj + all-reduce: fp32 sum (rank order) of the ranks' bf16 partials, identical bits everywhere
        flat = out.reshape(B, -1)
        got = tp_attn.forward(q0, kv, vv, kn0, vn0, cache_seqlens=cs, cache_batch_idx=batch_idx,
                              softmax_scale=scale, causal=True).clone()
        part = (flat.float() @ w_o.float()).to(DTYPE)
        parts = [torch.empty_like(part) for _ in range(world)]
        dist.all_gather(parts, part)
        acc = torch.zeros_like(part, dtype=torch.float32)
        for p in parts:
            acc += p.float()
        want_ar = acc.to(DTYPE)
        sc = want_ar.float().abs().max().item()
        e = (got.float() - want_ar.float()).abs().max().item()
        mine = got.view(torch.int16).to(torch.int32)
        ref0 = mine.clone()
        dist.broadcast(ref0, 0)
        same = torch.tensor([1 if torch.equal(mine, ref0) else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        ok_ar = e <= 2 * ULP[DTYPE] * sc
        okt = torch.tensor([1 if ok_ar else 0], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        res["oproj_allreduce"] = {"ok": bool(okt.item()), "arrangement": args.tp_collective,
                                  "max_err_over_scale": round(e / sc, 6), "tolerance": "2 bf16 ulps of the tensor scale",
                                  "identical_bits_on_all_ranks": bool(same.item()), "world": world}
        if not okt.item() or (args.tp_collective != "nccl" and not same.item()):
            raise RuntimeError(f"parity_check failed for the o_proj + all-reduce: {res}")
    return res


# ----------------------------------------------------------------------------- extras ---

def timed_ms(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def extra_prefill(att, va, dev, wl) -> dict:
    """configs[2]: Yi-6B-200K shapes (Hq 32, Hkv 4, D 128), chunked prefill of a 128K context, one
    layer, K/V in a vAttention tensor with fi_vattn_256kb page bookkeeping.  Per chunk: cache_flat +
    causal attention over everything cached so far.  FLOPs (causal-exact) = 4*Hq*D*(c*p + c(c+1)/2)."""
    Hq, Hkv, S = 32, 4, 131072
    kc, vc = va.init_kvcache(1, Hkv, D, 1, S, dev.index or 0, DTYPE, 256 << 10, False)
    va.reserve_physical_pages(2 * S * Hkv * D * 2 + (8 << 20))
    va.step([S], True)
    g = torch.Generator(device=dev).manual_seed(0)
    q = torch.randn(S, Hq, D, device=dev, generator=g).to(DTYPE)
    k = torch.randn(S, Hkv, D, device=dev, generator=g).to(DTYPE)
    v = torch.randn(S, Hkv, D, device=dev, generator=g).to(DTYPE)
    _, burst, sustained, _ = peaks()
    out = {"workload": "Yi-6B-200K shapes, 128K ctx chunked prefill, 1 layer, bf16, 256 KB logical pages; "
                       "whole prefill incl. cache_flat", "chunks": {}}
    for c in (2048, 512):
        def whole_prefill():
            for p in range(0, S, c):
                att.cache_flat(k[p:p + c], v[p:p + c], kc[0][p:], vc[0][p:], "auto")
                total = torch.tensor([p + c], dtype=torch.int32, device=dev)
                att.flash_attn_with_kvcache(q[p:p + c].unsqueeze(0), kc, vc, cache_seqlens=total, causal=True)
        ms = timed_ms(whole_prefill, 1, 2)
        flops = sum(4 * Hq * D * (c * p + c * (c + 1) // 2) for p in range(0, S, c))
        tf = flops / (ms * 1e-3) / 1e12
        out["chunks"][str(c)] = {"tflops": round(tf, 1), "ms_per_prefill": round(ms, 2),
                                 "frac_of_sustained": round(tf / sustained, 4), "frac_of_burst": round(tf / burst, 4)}
    out["tflops"] = out["chunks"]["2048"]["tflops"]
    out["frac_of_sustained"] = out["chunks"]["2048"]["frac_of_sustained"]
    out["chunk"], out["ctx"] = 2048, S
    out["peaks_tflops"] = {"burst": burst, "sustained": sustained}
    return out


def extra_pod(att, va, dev, wl) -> dict:
    """configs[3] (8 x 16K prefill + 56 x 4K decode, Llama-3-8B, fp16) and the balanced hybrid batch the
    POD wrapper issues (one 2048-token chunk at 16K + 64 decodes at 16K): the fused call vs the two
    calls back to back."""
    Hq, Hkv = 32, 8
    dtype = torch.float16
    hbm, burst, _, _ = peaks()
    res = {}
    for tag, (Bp, Sp, Sq, Bd, Sd) in (("configs3_8x16k_56x4k", (8, 16384, 16384, 56, 4096)),
                                       ("hybrid_1x2048at16k_64x16k", (1, 16384, 2048, 64, 16384))):
        g = torch.Generator(device=dev).manual_seed(0)
        q_p = torch.randn(Bp, Sq, Hq, D, device=dev, generator=g).to(dtype)
        kc_p = torch.randn(Bp, Sp, Hkv, D, device=dev, generator=g).to(dtype)
        vc_p = torch.randn(Bp, Sp, Hkv, D, device=dev, generator=g).to(dtype)
        lens_p = torch.full((Bp,), Sp, dtype=torch.int32, device=dev)
        q_d = torch.randn(Bd, 1, Hq, D, device=dev, generator=g).to(dtype)
        kc_d = torch.randn(Bd, Sd, Hkv, D, device=dev, generator=g).to(dtype)
        vc_d = torch.randn(Bd, Sd, Hkv, D, device=dev, generator=g).to(dtype)
        kn = torch.randn(Bd, 1, Hkv, D, device=dev, generator=g).to(dtype)
        vn = torch.randn(Bd, 1, Hkv, D, device=dev, generator=g).to(dtype)
        lens_d = torch.full((Bd,), Sd - 1, dtype=torch.int32, device=dev)
        idx = torch.randperm(Bd, device=dev, generator=g).int()

        def run_p():
            return att.flash_attn_with_kvcache(q_p, kc_p, vc_p, cache_seqlens=lens_p, causal=True)

        def run_d():
            return att.flash_attn_with_kvcache(q_d, kc_d, vc_d, kn, vn, cache_seqlens=lens_d,
                                               cache_batch_idx=idx, causal=True)

        def run_serial():
            run_p()
            run_d()

        def run_fused():
            return att.true_fused_attn_with_kvcache(q_p, kc_p, vc_p, q_d, kc_d, vc_d, kn, vn, causal=True,
                                                    cache_seqlens_p=lens_p, cache_seqlens_d=lens_d,
                                                    cache_batch_idx=idx, fused_params=15)

        it = 3 if Bp > 1 else 20
        t_p, t_d = timed_ms(run_p, 1, it), timed_ms(run_d, 3, 20)
        t_s, t_f = timed_ms(run_serial, 1, it), timed_ms(run_fused, 1, it)
        o_p, o_d = run_fused()
        # POD's contract (pod_attn/tests/attn_sweep.py:82-97): each output equals the separate call's
        s_p, s_d = run_p(), run_d()
        dmax = max((o_p.float() - s_p.float()).abs().max().item() / max(s_p.float().abs().max().item(), 1e-30),
                   (o_d.float() - s_d.float()).abs().max().item() / max(s_d.float().abs().max().item(), 1e-30))
        if dmax > 1e-3:
            raise RuntimeError(f"POD fused call differs from the separate calls: {dmax:.3e} of scale ({tag})")
        flops = Bp * 4 * Hq * D * (Sq * (Sp - Sq) + Sq * (Sq + 1) // 2)
        dbytes = 2 * 2 * Hkv * D * Bd * Sd
        res[tag] = {"prefill_ms": round(t_p, 3), "decode_ms": round(t_d, 4), "serial_ms": round(t_s, 3),
                    "fused_ms": round(t_f, 3), "speedup": round(t_s / t_f, 4),
                    "roofline_ms": round(max(flops / (burst * 1e12), dbytes / (hbm * 1e9)) * 1e3, 3),
                    "prefill_tflops": round(flops / (t_p * 1e-3) / 1e12, 1),
                    "decode_gbps": round(dbytes / (t_d * 1e-3) / 1e9, 1),
                    "fused_vs_separate_calls_max_diff_over_scale": round(dmax, 6)}
        del q_p, kc_p, vc_p, q_d, kc_d, vc_d
        torch.cuda.empty_cache()
    c3 = res["configs3_8x16k_56x4k"]
    return {"workload": "Llama-3-8B shapes fp16, true_fused_attn_with_kvcache(fused_params=15) vs the two calls",
            "serial_ms": c3["serial_ms"], "fused_ms": c3["fused_ms"], "speedup": c3["speedup"],
            "roofline_ms": c3["roofline_ms"], **res}


def extra_fa_vattn(att, va, dev, wl) -> dict:
    """The reference's GPU dispatch target on this box: flash_attn.flash_attn_with_kvcache over vAttention
    virtual tensors of the same shapes (decode32k: 2 timed steps; prefill: configs[2], chunk 2048)."""
    from flash_attn import flash_attn_with_kvcache as fa
    import flash_attn
    B, CTX, HQ, HKV, LAYERS = wl.batch, wl.ctx, wl.hq, wl.hkv, wl.layers
    n_res = 2
    tensors = va.init_kvcache(n_res, HKV, D, B, CTX, dev.index or 0, DTYPE, PAGE, False)
    va.reserve_physical_pages(n_res * 2 * B * CTX * HKV * D * 2)
    W, K = 1, 2
    start = CTX - (W + K) - 1
    lens = [start] * B
    va.step_async(lens)
    g = torch.Generator(device=dev).manual_seed(1234)
    for t in tensors:
        for b in range(B):
            t[b, :start + 4].normal_(generator=g)
    batch_idx = torch.randperm(B, generator=torch.Generator().manual_seed(0)).int().to(dev)
    q = torch.randn(LAYERS, B, 1, HQ, D, device=dev, generator=g).to(DTYPE)
    kn = torch.randn(LAYERS, B, 1, HKV, D, device=dev, generator=g).to(DTYPE)
    vn = torch.randn(LAYERS, B, 1, HKV, D, device=dev, generator=g).to(DTYPE)

    def one_step(lens_now):
        new = [n + 1 for n in lens_now]
        va.step_async(new)
        sl = torch.full((B,), lens_now[0], dtype=torch.int32, device=dev)
        for layer in range(LAYERS):
            fa(q[layer], tensors[layer % n_res][:, :lens_now[0] + 1], tensors[n_res + layer % n_res][:, :lens_now[0] + 1],
               kn[layer], vn[layer], cache_seqlens=sl, cache_batch_idx=batch_idx, softmax_scale=D ** -0.5, causal=True)
        return new

    for _ in range(W):
        lens = one_step(lens)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        lens = one_step(lens)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    hbm, _, sustained, _ = peaks()
    gbps = algorithmic_bytes(sum(lens), HQ, HKV, B) / (ms / K / LAYERS * 1e-3) / 1e9
    out = {"library": f"flash_attn {flash_attn.__version__} over vAttention tensors (same shapes, same box)",
           "tokens_s": round(B * K / (ms / 1e3), 2), "ms_per_layer_call": round(ms / K / LAYERS, 4),
           "approx_gbps": round(gbps, 1), "frac_of_measured_copy_peak": round(gbps / hbm, 4)}
    va.cleanup()
    # configs[2] prefill through the library
    Hq, Hkv, S, c = 32, 4, 131072, 2048
    kc, vc = va.init_kvcache(1, Hkv, D, 1, S, dev.index or 0, DTYPE, PAGE, False)
    va.reserve_physical_pages(2 * S * Hkv * D * 2 + (8 << 20))
    va.step([S], True)
    qq = torch.randn(S, Hq, D, device=dev, generator=g).to(DTYPE)
    k = torch.randn(S, Hkv, D, device=dev, generator=g).to(DTYPE)
    v = torch.randn(S, Hkv, D, device=dev, generator=g).to(DTYPE)

    def whole_prefill():
        for p in range(0, S, c):
            att.cache_flat(k[p:p + c], v[p:p + c], kc[0][p:], vc[0][p:], "auto")
            total = torch.tensor([p + c], dtype=torch.int32, device=dev)
            fa(qq[p:p + c].unsqueeze(0), kc, vc, cache_seqlens=total, causal=True)

    ms = timed_ms(whole_prefill, 1, 1)
    flops = sum(4 * Hq * D * (c * p + c * (c + 1) // 2) for p in range(0, S, c))
    out["prefill_tflops"] = round(flops / (ms * 1e-3) / 1e12, 1)
    out["prefill_frac_of_sustained"] = round(out["prefill_tflops"] / sustained, 4)
    return out


# -------------------------------------------------------------------------- reference ---

def cpu_unit_seconds(wl: Workload, n_seqs: int, threads: int, reps: int = 1) -> float:
    """Seconds for ONE (sequence, layer) unit of the workload on the CPU: torch SDPA decode over
    ctx keys, bf16 K/V, GQA handled by SDPA itself (enable_gqa: no materialised copy of K/V) -- the
    reference's CPU-runnable path, BASELINE configs[0] scaled to the workload's context."""
    from oracle import attention_ref as ref
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    q = torch.randn(n_seqs, 1, wl.hq, D, generator=g).to(DTYPE)
    k = torch.randn(n_seqs, wl.ctx, wl.hkv, D, generator=g).to(DTYPE)
    v = torch.randn(n_seqs, wl.ctx, wl.hkv, D, generator=g).to(DTYPE)
    ref.sdpa_decode_cpu(q[:1], k[:1], v[:1], D ** -0.5)  # warm up the thread pool
    t0 = time.perf_counter()
    for _ in range(reps):
        ref.sdpa_decode_cpu(q, k, v, D ** -0.5)
    return (time.perf_counter() - t0) / (reps * n_seqs)


def cpu_baseline(wl: Workload, sample_seqs: int = 2, budget_s: float = 20.0) -> dict:
    threads = os.cpu_count() or 1
    t_unit = cpu_unit_seconds(wl, sample_seqs, threads)
    reps = max(1, min(8, int(budget_s / max(t_unit * sample_seqs, 1e-3)) - 1))
    if reps > 1:
        t_unit = cpu_unit_seconds(wl, sample_seqs, threads, reps)
    return {"value": round(1.0 / (wl.layers * t_unit), 4), "unit": "tokens/s", "cores": threads,
            "kind": "port",
            "sample": f"torch SDPA (CPU, bf16, enable_gqa) on {sample_seqs} of the {wl.batch} sequences x 1 of "
                      f"{wl.layers} layers at {wl.ctx // 1024}K ctx, x{reps}; tokens/s = {wl.batch} / ({wl.layers} layers * "
                      f"{wl.batch} seqs * {t_unit * 1e3:.1f} ms per seq-layer)"}


def run_reference(args):
    wl = workload_from(args)
    rank, _, world = rank_info()
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    K, W = args.steps, args.warmup
    n = args.cpu_sample_seqs
    for _ in range(min(W, 1)):
        cpu_unit_seconds(wl, n, threads)
    t0 = time.perf_counter()
    units = 0.0
    for _ in range(K):
        units += cpu_unit_seconds(wl, n, threads) * n
    wall = time.perf_counter() - t0
    t_unit = units / (K * n)
    value = 1.0 / (wl.layers * t_unit)
    line = {"impl": "reference", "metric": f"decode tokens/s @{wl.ctx // 1024}K ctx ({wl.model} attention path)",
            "value": round(value, 4), "unit": "tokens/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": round(wall / K * 1e3, 2), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic N(0,1)",
            "config": {"workload": wl.name,
                       "shapes": f"B{wl.batch} Hq{wl.hq} Hkv{wl.hkv} D{D} L{wl.layers} ctx{wl.ctx} hidden{wl.hidden}",
                       "backend": "reference CPU path: torch SDPA on the host cores (attention only); each step is a "
                                  f"bounded sample of {n} (sequence, layer) units of the {wl.batch} x {wl.layers} in one "
                                  "decode iteration, extrapolated linearly"},
            "cpu_baseline": {"value": round(value, 4), "unit": "tokens/s", "cores": threads, "kind": "port",
                             "sample": f"{n} seq-layer units per step, {t_unit * 1e3:.1f} ms each"},
            "e2e": {"value": round(value, 4), "unit": "tokens/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- fa_vattn ---

def run_fa_vattn(args):
    """The reference's own GPU path on this box: ITS vattention extension (compiled unmodified from the
    original project's vattention/vattention.cu into oracle/_ref by oracle/Makefile) allocates the virtual
    tensors and maps the pages; flash_attn.flash_attn_with_kvcache (the library its wrapper dispatches
    to) attends over them.  A comparison arm; nothing of the product is on this path."""
    import glob
    import importlib.util
    from flash_attn import flash_attn_with_kvcache
    wl = workload_from(args)
    B, CTX, HQ, HKV, LAYERS = wl.batch, wl.ctx, wl.hq, wl.hkv, wl.layers
    dev = torch.device("cuda", 0)
    torch.zeros(1, device=dev)
    cands = glob.glob(str(ROOT / "oracle" / "_ref" / "vattention_ref*.so"))
    if cands:
        spec = importlib.util.spec_from_file_location("vattention_ref", cands[0])
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
        alloc = "reference vattention extension (oracle/_ref, compiled unmodified)"
    else:
        from vattention_b200 import vattention as ref
        alloc = "vattention_b200 allocator (oracle/_ref not built)"
    n_res = args.resident_layers
    K, W = args.steps, args.warmup
    start_len = CTX - (W + K) - 2
    tensors = ref.init_kvcache(n_res, HKV, D, B, CTX, 0, DTYPE, PAGE, False)
    ref.reserve_physical_pages(n_res * 2 * B * CTX * HKV * D * 2)
    seq_lens = [start_len] * B
    ref.step(seq_lens, False)        # synchronous: every page of the start state mapped on return
    g = torch.Generator(device=dev).manual_seed(1234)
    for t in tensors:
        for b in range(B):
            t[b, :start_len + 8].normal_(generator=g)
    batch_idx = torch.randperm(B, generator=torch.Generator().manual_seed(0)).int().to(dev)
    q = torch.randn(LAYERS, B, 1, HQ, D, device=dev, generator=g).to(DTYPE)
    kn = torch.randn(LAYERS, B, 1, HKV, D, device=dev, generator=g).to(DTYPE)
    vn = torch.randn(LAYERS, B, 1, HKV, D, device=dev, generator=g).to(DTYPE)

    def one_step(lens_now):
        new_lens = [n + 1 for n in lens_now]
        ref.step_async(new_lens)
        sl = torch.full((B,), lens_now[0], dtype=torch.int32, device=dev)
        for layer in range(LAYERS):
            flash_attn_with_kvcache(q[layer], tensors[layer % n_res][:, :lens_now[0] + 1],
                                    tensors[n_res + layer % n_res][:, :lens_now[0] + 1], kn[layer], vn[layer],
                                    cache_seqlens=sl, cache_batch_idx=batch_idx, softmax_scale=D ** -0.5,
                                    causal=True)
        return new_lens

    for _ in range(W):
        seq_lens = one_step(seq_lens)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        seq_lens = one_step(seq_lens)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    hbm, _, _, _ = peaks()
    gbps = algorithmic_bytes(sum(seq_lens), HQ, HKV, B) / (ms / K / LAYERS * 1e-3) / 1e9
    print(json.dumps({"impl": "fa_vattn", "allocator": alloc, "attention": "flash_attn.flash_attn_with_kvcache",
                      "value": round(B * K / (ms / 1e3), 2), "unit": "tokens/s", "steps": K, "warmup": W,
                      "config": {"workload": wl.name}, "ms_per_layer_call": round(ms / K / LAYERS, 4),
                      "approx_gbps_incl_all_kernels": round(gbps, 1), "frac_of_peak": round(gbps / hbm, 4)}),
          flush=True)
    os._exit(0)      # the reference extension has no re-entrant cleanup; leave without running destructors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "fa_vattn"])
    ap.add_argument("--workload", default="decode32k", choices=["decode32k", "tp70b"])
    ap.add_argument("--ctx", type=int, default=0, help="context length (default 32768; tp70b: 32768 | 65536 | 131072)")
    ap.add_argument("--resident-layers", type=int, default=4)
    # N > 1: "fused" = our single GEMM + all-reduce kernel (csrc/oproj_allreduce.cu) inside the CUDA graph;
    # "peer" = cuBLAS + our one-shot all-reduce kernel (eager only: its epoch is a host-side argument);
    # "nccl" = cuBLAS + NCCL
    ap.add_argument("--tp-collective", default="fused", choices=["fused", "peer", "nccl"])
    ap.add_argument("--no-graph", "--no-tp-graph", dest="graph", action="store_false",
                    help="launch the layer-calls eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the prefill / pod / fa_vattn legs (N = 1)")
    ap.add_argument("--cpu-sample-seqs", type=int, default=2)
    ap.add_argument("--cpu-budget-s", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (float32): "
                         "block_out [layer-calls, batch, hidden], k_appended / v_appended [resident layers, "
                         "batch, kv heads, head dim]")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "fa_vattn":
        run_fa_vattn(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
