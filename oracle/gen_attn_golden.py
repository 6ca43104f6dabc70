"""Generate tests/golden/attn_*.pt: outputs of flash_attn.flash_attn_with_kvcache (the
un-vendored dependency the reference dispatches to; installed 2.8.3, reference pin
2.5.9.post1) on small seeded inputs.  Runs on the GPU box:
    python oracle/gen_attn_golden.py [outdir]      (default gpurun_out/golden)
Each file stores the inputs (so the fixture does not depend on RNG reproducibility), the
library's output and the rows its append wrote into the caches (`with_appended` rebuilds the caches
after the call; the rest of them is unchanged, which is checked here).  TEST INFRASTRUCTURE ONLY.
"""
import os
import sys
import zlib

import torch

CASES = [
    # name, B, Sq, Hq, Hkv, D, Sk, dtype, append, causal, slots
    ("decode_gqa4_bf16", 3, 1, 8, 2, 128, 160, torch.bfloat16, True, True, 4),
    ("decode_mha_fp16", 2, 1, 4, 4, 128, 96, torch.float16, True, True, 2),
    ("decode_d64_fp16", 2, 1, 6, 2, 64, 130, torch.float16, True, False, 3),
    ("prefill_chunk_bf16", 1, 48, 8, 2, 128, 176, torch.bfloat16, False, True, 1),
    ("prefill_square_fp16", 2, 40, 4, 2, 128, 40, torch.float16, False, True, 2),
    ("prefill_masked_rows_fp16", 1, 24, 4, 4, 64, 64, torch.float16, False, True, 1),
    # rotary cases (name prefix rope_): (interleaved, rotary_dim) in ROPE below
    ("rope_decode_neox_bf16", 3, 1, 8, 2, 128, 160, torch.bfloat16, True, True, 4),
    ("rope_decode_gptj_fp16", 2, 1, 4, 4, 128, 96, torch.float16, True, True, 2),
    ("rope_append4_causal_partial_fp16", 2, 4, 4, 2, 128, 80, torch.float16, True, True, 3),
    ("rope_append4_noncausal_bf16", 2, 4, 4, 2, 64, 80, torch.bfloat16, True, False, 2),
]
ROPE = {"rope_decode_neox_bf16": (False, 128), "rope_decode_gptj_fp16": (True, 128),
        "rope_append4_causal_partial_fp16": (False, 64), "rope_append4_noncausal_bf16": (True, 32)}


def with_appended(cache, rows, lens, idx):
    """A copy of `cache` [slots, Sk, Hkv, D] with rows[b] written at rows [lens[b], lens[b] + n) of
    batch row b's slot (idx[b], or b without an index); `rows` [B, n, Hkv, D] or None."""
    out = cache.clone()
    if rows is not None:
        slots = range(rows.shape[0]) if idx is None else idx.tolist()
        for b, (s, n) in enumerate(zip(slots, lens.tolist())):
            out[s, n:n + rows.shape[1]] = rows[b]
    return out


def appended_rows(before, after, lens, idx, n_new):
    """The rows a call appended to a cache (None without an append); raises if it changed anything
    else."""
    rows = None
    if n_new:
        slots = range(len(lens)) if idx is None else idx.tolist()
        rows = torch.stack([after[s, n:n + n_new] for s, n in zip(slots, lens.tolist())])
    if not torch.equal(with_appended(before, rows, lens, idx), after):
        raise RuntimeError("the call changed cache rows outside the appended ones")
    return rows


def main(outdir):
    from flash_attn import flash_attn_with_kvcache
    import flash_attn
    os.makedirs(outdir, exist_ok=True)
    for name, B, Sq, Hq, Hkv, D, Sk, dtype, append, causal, slots in CASES:
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        q = torch.randn(B, Sq, Hq, D, generator=g).to(dtype)
        kc = torch.randn(slots, Sk, Hkv, D, generator=g).to(dtype)
        vc = torch.randn(slots, Sk, Hkv, D, generator=g).to(dtype)
        n_new = Sq if append else 0
        if name == "prefill_masked_rows_fp16":
            lens = torch.tensor([10], dtype=torch.int32)          # Sq > Lk: leading rows fully masked
        elif append:
            lens = torch.randint(1, Sk - n_new + 1, (B,), generator=g).int()
            lens[0] = Sk - n_new
        else:
            lens = torch.randint(Sq, Sk + 1, (B,), generator=g).int()
        kn = torch.randn(B, n_new, Hkv, D, generator=g).to(dtype) if append else None
        vn = torch.randn(B, n_new, Hkv, D, generator=g).to(dtype) if append else None
        idx = torch.randperm(slots, generator=g)[:B].int() if slots != B else None
        dev = lambda t: None if t is None else t.cuda()
        kc_d, vc_d = dev(kc), dev(vc)
        cos = sin = None
        interleaved = True
        if name in ROPE:
            interleaved, rd = ROPE[name]
            ang = torch.rand(Sk, rd // 2, generator=g) * 6.283
            cos, sin = torch.cos(ang).to(dtype), torch.sin(ang).to(dtype)
        out = flash_attn_with_kvcache(dev(q), kc_d, vc_d, dev(kn), dev(vn), rotary_cos=dev(cos),
                                      rotary_sin=dev(sin), cache_seqlens=dev(lens),
                                      cache_batch_idx=dev(idx), causal=causal,
                                      rotary_interleaved=interleaved)
        torch.cuda.synchronize()
        torch.save({"name": name, "source": f"flash_attn {flash_attn.__version__} on {torch.cuda.get_device_name(0)}",
                    "q": q, "k_cache": kc, "v_cache": vc, "k": kn, "v": vn, "cache_seqlens": lens,
                    "cache_batch_idx": idx, "causal": causal, "out": out.cpu(),
                    "rotary_cos": cos, "rotary_sin": sin, "rotary_interleaved": interleaved,
                    "k_cache_appended": appended_rows(kc, kc_d.cpu(), lens, idx, n_new),
                    "v_cache_appended": appended_rows(vc, vc_d.cpu(), lens, idx, n_new)},
                   os.path.join(outdir, f"attn_{name}.pt"))
        print(name, tuple(out.shape))


if __name__ == "__main__":
    here = os.path.dirname(os.path.abspath(__file__))
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(here), "gpurun_out", "golden"))
