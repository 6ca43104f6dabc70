"""Drop-in proof for the wrapper call sites (north_star: "keeping ... the sarathi
vattention_flashattention_wrapper / vattention_flashinfer_wrapper call sites so it is a drop-in").

1. tests/golden/wrapper_call_trace.json was recorded from the reference's three wrapper files and
   its base class, loaded UNMODIFIED with importlib over vattention_b200.dropin's module shims
   (`vattention`, `flash_attn`, `flashinfer`, `pod_attn`, `sarathi.cache_ops`) plus stubs for the
   parts of sarathi outside the hot path (config, metrics, logger, sequence).  The shims are given
   CPU stand-ins for the operators that (a) bind every call to the PRODUCT operator's Python
   signature (so a call our operator would reject fails) and (b) compute with the oracle.  One
   scheduler iteration -- a prefill chunk plus three decodes -- had to produce the oracle's output
   and the cache contents; the exact sequence of operator calls (names, shapes, keyword set) is the
   golden.
2. This package's wrapper mirrors (vattention_b200/wrappers.py) must emit the same call trace as
   that golden and the same outputs -- the mirrors behave like the reference's files.
3. On the GPU: the shims are installed with the REAL operators and the same iteration runs on
   cuda:0 through names imported the way the reference imports them; outputs against the oracle.

Regenerate the golden from a checkout of the original project (it runs the check of 1 as well),
from the repository root:
    PYTHONPATH=. python tests/test_dropin_reference_wrappers.py <checkout>
"""
import enum
import importlib.util
import inspect
import json
import sys
import types
from pathlib import Path

import pytest
import torch

from oracle import attention_ref as ref
from vattention_b200 import dropin

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden" / "wrapper_call_trace.json"
WRAPPERS = {
    "fa_vattn": ("vattention_flashattention_wrapper.py", "VAttentionFlashAttentionWrapper"),
    "fi_vattn": ("vattention_flashinfer_wrapper.py", "VAttentionFlashInferWrapper"),
    "fa_pod": ("vattention_flashattention_pod_wrapper.py", "VAttentionFlashAttentionPODWrapper"),
}


# ---- minimal stand-ins for sarathi objects outside the hot path ----------------------------------
class Seq:
    def __init__(self, seq_id, prompt_len, processed=0, generated=0):
        self.seq_id, self.prompt_len, self.processed, self.generated = seq_id, prompt_len, processed, generated

    def get_next_prompt_chunk_len(self, chunk):
        return min(chunk, self.prompt_len - self.processed)

    def get_num_prompt_tokens_processed(self):
        return self.processed

    def get_len(self):
        return self.prompt_len + self.generated


class MD:
    def __init__(self, seq, is_prompt, chunk=0):
        self.seq, self.is_prompt, self.prompt_chunk_len = seq, is_prompt, chunk


class ModelConfig:
    def __init__(self, hq, hkv, d, dtype):
        self.hq, self.hkv, self.d, self.dtype = hq, hkv, d, dtype

    def get_num_q_heads(self, parallel_config):
        return self.hq

    def get_num_kv_heads(self, parallel_config):
        return self.hkv

    def get_head_size(self):
        return self.d


def sarathi_stubs():
    """Modules the wrapper files import that are NOT on the hot path."""
    class _Anything(enum.Enum):
        pass

    class OperationMetrics:
        def __getattr__(self, name):
            return name
    om = OperationMetrics()

    class CudaTimer:
        def __init__(self, *a, **k):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    class _Logger:
        def __getattr__(self, name):
            return lambda *a, **k: None

    mods = {}

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        m.__path__ = []
        mods[name] = m
        return m

    mod("sarathi")
    mod("sarathi.config", ModelConfig=ModelConfig, ParallelConfig=object)
    mod("sarathi.core")
    mod("sarathi.core.datatypes")
    mod("sarathi.core.datatypes.sequence", SequenceMetadata=MD)
    mod("sarathi.logger", init_logger=lambda name: _Logger())
    mod("sarathi.metrics")
    mod("sarathi.metrics.constants", OperationMetrics=om)
    mod("sarathi.metrics.cuda_timer", CudaTimer=CudaTimer)
    mod("sarathi.model_executor")
    mod("sarathi.model_executor.attention")
    return mods


# ---- CPU stand-ins for the operators: product signature + oracle arithmetic + call recording ------
def describe(x):
    if isinstance(x, torch.Tensor):
        return ["tensor", list(x.shape), str(x.dtype).replace("torch.", "")]
    if isinstance(x, (bool, int, str)) or x is None:
        return x
    if isinstance(x, float):
        return round(x, 6)
    return type(x).__name__


class RecordingOps:
    """Operator namespace with the product's call surface (signatures taken from
    vattention_b200.attention at call time), oracle arithmetic, and a trace of the calls."""

    def __init__(self):
        from vattention_b200 import attention as product
        self.product = product
        self.trace = []

    def _bind(self, name, args, kwargs):
        sig = inspect.signature(getattr(self.product, name))
        bound = sig.bind(*args, **kwargs)          # TypeError if the product could not take this call
        self.trace.append({"op": name,
                           "args": {k: describe(v) for k, v in bound.arguments.items()}})
        return bound.arguments

    def flash_attn_with_kvcache(self, *args, **kwargs):
        a = self._bind("flash_attn_with_kvcache", args, kwargs)
        if a.get("block_table") is not None:
            raise RuntimeError("block_table is not supported")
        return ref.attn_with_kvcache_ref(a["q"], a["k_cache"], a["v_cache"], a.get("k"), a.get("v"),
                                         a.get("cache_seqlens"), a.get("cache_batch_idx"),
                                         a.get("softmax_scale"), a.get("causal", False))

    def single_prefill_with_kv_cache(self, *args, **kwargs):
        a = self._bind("single_prefill_with_kv_cache", args, kwargs)
        return ref.single_prefill_ref(a["q"], a["k"], a["v"], a.get("causal", False), a.get("sm_scale"))

    def true_fused_attn_with_kvcache(self, *args, **kwargs):
        a = self._bind("true_fused_attn_with_kvcache", args, kwargs)
        o_p = o_d = None
        if a["q_p"] is not None:
            o_p = ref.attn_with_kvcache_ref(a["q_p"], a["k_cache_p"], a["v_cache_p"],
                                            cache_seqlens=a.get("cache_seqlens_p"),
                                            softmax_scale=a.get("softmax_scale"), causal=a.get("causal", False))
        if a["q_d"] is not None:
            o_d = ref.attn_with_kvcache_ref(a["q_d"], a["k_cache_d"], a["v_cache_d"], a.get("k"), a.get("v"),
                                            a.get("cache_seqlens_d"), a.get("cache_batch_idx"),
                                            a.get("softmax_scale"), a.get("causal", False))
        return o_p, o_d

    def cache_flat(self, *args, **kwargs):
        a = self._bind("cache_flat", args, kwargs)
        ref.cache_flat_ref(a["key"], a["value"], a["k_cache"], a["v_cache"])


def load_reference_wrapper(kind, ref_attn):
    """The reference's wrapper class, from its unmodified file in `ref_attn` (module shims must be
    installed)."""
    base = ref_attn / "base_attention_wrapper.py"
    name = "sarathi.model_executor.attention.base_attention_wrapper"
    spec = importlib.util.spec_from_file_location(name, base)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    fname, cls = WRAPPERS[kind]
    name = "sarathi.model_executor.attention." + fname[:-3]
    spec = importlib.util.spec_from_file_location(name, ref_attn / fname)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return getattr(m, cls)


def mixed_batch(kind, dtype=torch.float32, device="cpu", D=64):
    """One prefill chunk and three decodes, flat [tokens, H*D] tensors (the model runner's layout)."""
    g = torch.Generator().manual_seed(0)
    Hq, Hkv, B, ctx = 4, 2, 5, 256
    kc = torch.randn(B, ctx, Hkv, D, generator=g).to(dtype)
    vc = torch.randn(B, ctx, Hkv, D, generator=g).to(dtype)
    # the reference's POD wrapper hands cache_flat the un-offset cache (pod_wrapper.py:153-158): only
    # its first chunk is well defined, so the POD case prefills from position 0
    done = 0 if kind == "fa_pod" else 64
    p = Seq(1, 200, processed=done)
    decs = [Seq(2, 50, 50, 3), Seq(3, 120, 120, 1), Seq(4, 7, 7, 9)]
    mds = [MD(decs[0], False), MD(p, True, 32), MD(decs[1], False), MD(decs[2], False)]
    q = torch.randn(35, Hq * D, generator=g).to(dtype)
    k = torch.randn(35, Hkv * D, generator=g).to(dtype)
    v = torch.randn(35, Hkv * D, generator=g).to(dtype)
    slots = {1: 3, 2: 0, 3: 4, 4: 1}
    dev = torch.device(device)
    return (Hq, Hkv, D), (kc.to(dev), vc.to(dev)), mds, (q.to(dev), k.to(dev), v.to(dev)), slots, p, decs, done


def expected(kind, dims, caches, qkv, slots, p, decs, done, scale):
    Hq, Hkv, D = dims
    kc, vc = caches[0].clone().cpu(), caches[1].clone().cpu()
    q, k, v = [t.cpu() for t in qkv]
    out = torch.empty_like(q)
    sp = slots[p.seq_id]
    kc[sp, done:done + 32] = k[:32].view(32, Hkv, D)
    vc[sp, done:done + 32] = v[:32].view(32, Hkv, D)
    # fi_vattn's prefill goes through single_prefill_with_kv_cache without a scale: 1/sqrt(D)
    want_p = ref.attn_with_kvcache_ref(q[:32].view(1, 32, Hq, D), kc[sp:sp + 1], vc[sp:sp + 1],
                                       cache_seqlens=torch.tensor([done + 32], dtype=torch.int32),
                                       softmax_scale=scale, causal=True)
    out[:32] = want_p.reshape(32, -1)
    for j, s in enumerate(decs):
        sl, L0 = slots[s.seq_id], s.get_len() - 1
        kc[sl, L0] = k[32 + j].view(Hkv, D)
        vc[sl, L0] = v[32 + j].view(Hkv, D)
        want = ref.attn_with_kvcache_ref(q[32 + j].view(1, 1, Hq, D), kc[sl:sl + 1], vc[sl:sl + 1],
                                         cache_seqlens=torch.tensor([L0 + 1], dtype=torch.int32),
                                         softmax_scale=scale)
        out[32 + j] = want.reshape(-1)
    return out, kc, vc


def run_iteration(wrapper, kind, batch, device="cpu"):
    dims, caches, mds, qkv, slots, p, decs, done = batch
    Hq, Hkv, D = dims
    scale = D ** -0.5
    b_idx = torch.tensor([slots[p.seq_id]] + [slots[s.seq_id] for s in decs], dtype=torch.int32, device=device)
    wrapper.set_batch_idx(b_idx, b_idx[1:])
    wrapper.begin_forward(mds)
    out = wrapper.forward(qkv[0], qkv[1], qkv[2], caches, softmax_scale=scale, layer_id=0)
    wrapper.end_forward()
    return out


def reference_trace_and_check(kind, ref_attn):
    ops = RecordingOps()
    saved = {n: sys.modules.get(n) for n in list(sarathi_stubs())}
    stubs = sarathi_stubs()
    sys.modules.update(stubs)
    try:
        with dropin.installed(ops=ops, allocator=types.SimpleNamespace()):
            cls = load_reference_wrapper(kind, ref_attn)
            batch = mixed_batch(kind)
            w = cls()
            w.init(ModelConfig(*batch[0], torch.float32), None, 0, torch.device("cpu"))
            out = run_iteration(w, kind, batch)
    finally:
        for n in list(sys.modules):
            if n == "sarathi" or n.startswith("sarathi."):
                del sys.modules[n]
        for n, m in saved.items():
            if m is not None:
                sys.modules[n] = m
    dims, caches, mds, qkv, slots, p, decs, done = batch
    want, kc, vc = expected(kind, dims, mixed_batch(kind)[1], qkv, slots, p, decs, done, dims[2] ** -0.5)
    assert torch.allclose(out, want, atol=1e-5), f"{kind}: unmodified reference wrapper over the shims != oracle"
    assert torch.equal(caches[0], kc) and torch.equal(caches[1], vc)
    return ops.trace


def mirror_trace_and_check(kind):
    from vattention_b200.wrappers import get_attention_wrapper_class
    ops = RecordingOps()
    batch = mixed_batch(kind)
    w = get_attention_wrapper_class(kind)(ops=ops).init(num_q_heads=batch[0][0], num_kv_heads=batch[0][1],
                                                        head_dim=batch[0][2], device=torch.device("cpu"))
    out = run_iteration(w, kind, batch)
    dims, caches, mds, qkv, slots, p, decs, done = batch
    want, kc, vc = expected(kind, dims, mixed_batch(kind)[1], qkv, slots, p, decs, done, dims[2] ** -0.5)
    assert torch.allclose(out, want, atol=1e-5)
    assert torch.equal(caches[0], kc) and torch.equal(caches[1], vc)
    return ops.trace


def normalise(trace):
    """What must agree between the reference's files and the mirrors: the operators called, in order,
    with the same tensor shapes and the same values for the arguments that change the arithmetic.
    (The mirrors skip arguments whose value is the operator's default.)"""
    keep = ("q", "k_cache", "v_cache", "k", "v", "cache_seqlens", "cache_batch_idx", "causal", "key", "value",
            "q_p", "k_cache_p", "v_cache_p", "q_d", "k_cache_d", "v_cache_d", "cache_seqlens_p", "cache_seqlens_d")
    out = []
    for c in trace:
        out.append({"op": c["op"], "args": {k: v for k, v in c["args"].items() if k in keep and v is not None}})
    return out


@pytest.mark.parametrize("kind", list(WRAPPERS))
def test_mirror_wrappers_make_the_reference_wrappers_calls(kind):
    golden = json.loads(GOLDEN.read_text())
    got = normalise(mirror_trace_and_check(kind))
    want = golden[kind]
    if kind == "fa_pod":
        # documented difference (wrappers.py): the mirror writes the chunk at row `processed`; with
        # processed == 0 (this case) the calls are identical
        pass
    assert got == want


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(WRAPPERS))
def test_shims_with_the_cuda_operators_match_the_oracle(kind):
    """The reference's import lines, executed against the installed shims, on cuda:0."""
    from vattention_b200.wrappers import get_attention_wrapper_class
    with dropin.installed():
        import flash_attn as fa_mod                     # noqa: F401 -- resolved to the shim
        from flash_attn import flash_attn_with_kvcache  # vattention_flashattention_wrapper.py:4
        from flashinfer import single_prefill_with_kv_cache  # vattention_flashinfer_wrapper.py:5
        import pod_attn as fused                        # vattention_flashattention_pod_wrapper.py:14
        from sarathi.cache_ops import cache_flat        # :12
        import vattention                               # :11
        ops = types.SimpleNamespace(flash_attn_with_kvcache=flash_attn_with_kvcache,
                                    single_prefill_with_kv_cache=single_prefill_with_kv_cache,
                                    true_fused_attn_with_kvcache=fused.true_fused_attn_with_kvcache,
                                    cache_flat=cache_flat)
        assert fa_mod.__version__ == "vattention_b200" and hasattr(vattention, "step_async")
    batch = mixed_batch(kind, dtype=torch.float16, device="cuda:0", D=128)
    dims = batch[0]
    w = get_attention_wrapper_class(kind)(ops=ops).init(num_q_heads=dims[0], num_kv_heads=dims[1], head_dim=dims[2],
                                                        device=torch.device("cuda:0"))
    out = run_iteration(w, kind, batch, device="cuda:0")
    torch.cuda.synchronize()
    _, caches, mds, qkv, slots, p, decs, done = batch
    fresh = mixed_batch(kind, dtype=torch.float16, device="cpu", D=128)
    want, kc, vc = expected(kind, dims, fresh[1], fresh[3], slots, p, decs, done, dims[2] ** -0.5)
    err = (out.float().cpu() - want.float()).abs().max().item()
    assert err <= 1e-3 * want.float().abs().max().item() + 2.0 ** -10 * want.float().abs().max().item()
    assert torch.equal(caches[0].cpu(), kc) and torch.equal(caches[1].cpu(), vc)


if __name__ == "__main__":
    attn_dir = Path(sys.argv[1]) / "sarathi-lean" / "sarathi" / "model_executor" / "attention"
    GOLDEN.write_text(json.dumps({k: normalise(reference_trace_and_check(k, attn_dir)) for k in WRAPPERS},
                                 indent=1))
    print("wrote", GOLDEN)
