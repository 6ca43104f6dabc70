"""GPU: the allocator against the real CUDA VMM driver.

* data written through one virtual tensor lands in physical pages and survives further growth;
* rows beyond the mapped prefix are genuinely unmapped (the kernels must never touch them);
* traces replayed on the real driver match the oracle bit for bit, and the snapshots the reference
  extension itself produced on a B200 (tests/golden/alloc_trace_*.json) as well;
* attention reads straight out of the virtual tensors.
"""
import ctypes
import json
from pathlib import Path

import pytest
import torch

from oracle import alloc_traces as T
from oracle import attention_ref as ref
from oracle.allocator_model import MB
from vattention_b200 import attention as att
from vattention_b200 import vattention as va

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(autouse=True)
def fresh():
    torch.zeros(1, device="cuda")  # the allocator needs torch's context (cudaInternal.h:19-25)
    yield
    va.cleanup()


def test_granularity_is_2mb_and_tensors_are_virtual():
    ts = va.init_kvcache(2, 8, 128, 4, 32768, 0, torch.bfloat16, 2 * MB, False)
    cfg = va.get_config()
    assert cfg["phys_granularity"] == 2 * MB
    assert len(ts) == 4 and tuple(ts[0].shape) == (4, 32768, 8, 128)
    assert ts[0].is_cuda and ts[0].dtype == torch.bfloat16 and ts[0].is_contiguous()
    assert ts[0].stride(0) * 2 == cfg["virt_buff_size_per_req"]
    free0 = torch.cuda.mem_get_info()[0]
    assert va.reserve_physical_pages(64 * MB) == 32
    assert free0 - torch.cuda.mem_get_info()[0] >= 60 * MB  # physical memory really reserved


def test_write_read_through_mapped_pages_and_growth():
    L, Hkv, D, B, ctx = 2, 8, 128, 3, 8192
    ts = va.init_kvcache(L, Hkv, D, B, ctx, 0, torch.float16, 2 * MB, False)
    va.reserve_physical_pages(128 * MB)
    tpp = va.get_config()["tokens_per_page"]
    lens = [tpp + 5, 0, 3]
    va.step(lens, True)
    for t_i, t in enumerate(ts):
        t[0, : lens[0]] = float(t_i + 1)
        t[2, : lens[2]] = float(-(t_i + 1))
    torch.cuda.synchronize()
    lens = [3 * tpp, 7, 3]
    va.step(lens, True)          # growth must keep what was written (pages stay mapped)
    for t_i, t in enumerate(ts):
        assert torch.all(t[0, : tpp + 5] == float(t_i + 1))
        assert torch.all(t[2, :3] == float(-(t_i + 1)))
        t[0, tpp + 5: 3 * tpp] = 9.0
        t[1, :7] = 5.0
    torch.cuda.synchronize()
    st = va.get_state()
    assert st["mapped_pages"] == [3, 1, 1]
    # distinct physical pages everywhere
    ids = [p for e in st["pagemap"] for p in e[3:]]
    assert len(ids) == len(set(ids)) == 5 * 2 * L


def backed_by_physical_memory(addr: int) -> bool:
    """Whether the driver has physical memory mapped at `addr` (cuMemRetainAllocationHandle fails
    for an address that is not mapped); asks the driver instead of touching the address."""
    cuda = ctypes.CDLL("libcuda.so.1")
    handle = ctypes.c_ulonglong()
    if cuda.cuMemRetainAllocationHandle(ctypes.byref(handle), ctypes.c_void_p(addr)) != 0:
        return False
    assert cuda.cuMemRelease(handle) == 0
    return True


def test_rows_beyond_the_mapped_prefix_are_unmapped():
    """Virtual addresses beyond the mapped prefix have no physical memory behind them (a kernel
    touching them would fault, not read zeros): proves the tensors are virtual and that kernels must
    respect the mapped prefix."""
    ts = va.init_kvcache(1, 8, 128, 2, 8192, 0, torch.float16, 2 * MB, False)
    va.reserve_physical_pages(16 * MB)
    va.step([10, 0], True)
    assert va.get_state()["mapped_pages"] == [1, 0]
    tpp = va.get_config()["tokens_per_page"]
    ts[0][0, :10] = 1.0
    torch.cuda.synchronize()
    assert torch.all(ts[0][0, :10] == 1.0)
    for t in ts:
        assert backed_by_physical_memory(t[0, 0].data_ptr())
        assert backed_by_physical_memory(t[0, tpp - 1].data_ptr())     # the rest of the first page
        assert not backed_by_physical_memory(t[0, tpp].data_ptr())     # request 0's second page
        assert not backed_by_physical_memory(t[1, 0].data_ptr())       # request 1 has no tokens


@pytest.mark.parametrize("name", T.TRACE_NAMES)
def test_traces_on_real_driver_match_oracle(name):
    mb, pb = T.ModelBackend(), T.ProductBackend(va, torch)
    concrete = T.expand(T.build_trace(name), mb)
    for op in concrete:
        pb(op)
    T.compare_snaps(pb.snaps, mb.snaps, f"product(cuda) vs oracle [{name}]")


@pytest.mark.parametrize("name", ["llama8b_async", "mega_async", "tight_pool_sync"])
def test_traces_match_live_reference(name):
    """The product on the real driver against the snapshots the reference extension produced for
    the same calls on a B200 (recorded by oracle/gen_alloc_golden.py)."""
    gold = json.loads((ROOT / "tests" / "golden" / f"alloc_trace_{name}.json").read_text())
    ref_snaps = [dict(s, op=o) for s, o in zip(gold["snaps"], gold["trace"])]
    mb, pb = T.ModelBackend(), T.ProductBackend(va, torch)
    concrete = T.expand(T.build_trace(name), mb)
    assert concrete == gold["trace"]
    for o in concrete:
        pb(o)
    T.compare_snaps(pb.snaps, ref_snaps, f"product(cuda) vs reference [{name}]")
    T.compare_snaps(mb.snaps, ref_snaps, f"oracle vs reference [{name}]")


@pytest.mark.parametrize("mega,page", [(False, 2 * MB), (True, 2 * MB), (False, 256 * 1024)])
def test_decode_attention_over_virtual_tensors(mega, page):
    """The fa_vattn flow end to end: allocator -> cache_flat prefill write -> decode with append,
    reading the virtual tensors with cache_batch_idx (wrapper.py:151-155,194-205).  The 256 KB case
    is the reference's fi_vattn_256kb page size: logical pages over 2 MiB physical chunks."""
    L, Hkv, D, Hq, B, ctx = 2, 4, 128, 16, 6, 16384
    dtype = torch.bfloat16
    ts = va.init_kvcache(L, Hkv, D, B, ctx, 0, dtype, page, mega)
    va.reserve_physical_pages(256 * MB)
    if mega:
        caches = [(ts[0][:, :, i], ts[1][:, :, i]) for i in range(L)]
    else:
        caches = list(zip(ts[:L], ts[L:]))
    g = torch.Generator().manual_seed(3)
    ctx_lens = [700, 2049, 33, 1500]
    rids = [va.alloc_new_batch_idx(n) for n in ctx_lens]
    lens = [0] * B
    for r, n in zip(rids, ctx_lens):
        lens[r] = n
    va.step_async(lens)
    host_k = {}
    for layer, (kc, vc) in enumerate(caches):
        for r, n in zip(rids, ctx_lens):
            k = torch.randn(n, Hkv, D, generator=g).to(dtype)
            v = torch.randn(n, Hkv, D, generator=g).to(dtype)
            host_k[(layer, r)] = (k, v)
            att.cache_flat(k.cuda(), v.cuda(), kc[r], vc[r], "auto")
    # one decode step: every sequence grows by one token
    lens = [n + 1 if n else 0 for n in lens]
    va.step_async(lens)
    q = torch.randn(len(rids), 1, Hq, D, generator=g).to(dtype)
    kn = torch.randn(len(rids), 1, Hkv, D, generator=g).to(dtype)
    vn = torch.randn(len(rids), 1, Hkv, D, generator=g).to(dtype)
    seqlens = torch.tensor(ctx_lens, dtype=torch.int32)
    idx = torch.tensor(rids, dtype=torch.int32)
    max_len = max(ctx_lens) + 1
    for layer, (kc, vc) in enumerate(caches):
        out = att.flash_attn_with_kvcache(q.cuda(), kc[:, :max_len], vc[:, :max_len], kn.cuda(), vn.cuda(),
                                          cache_seqlens=seqlens.cuda(), cache_batch_idx=idx.cuda(), causal=True)
        kref = torch.zeros(B, max_len, Hkv, D, dtype=dtype)
        vref = torch.zeros(B, max_len, Hkv, D, dtype=dtype)
        for r, n in zip(rids, ctx_lens):
            kref[r, :n], vref[r, :n] = host_k[(layer, r)]
        want = ref.attn_with_kvcache_ref(q, kref, vref, kn, vn, seqlens, idx, causal=True)
        err = (out.float().cpu() - want.float()).abs().max().item()
        assert err <= 1e-3 * want.float().abs().max().item() + 2 ** -7 * want.float().abs().max().item(), err
        for i, (r, n) in enumerate(zip(rids, ctx_lens)):  # the appended row is in the virtual tensor
            assert torch.equal(kc[r, n].cpu(), kn[i, 0])


def test_async_overlap_stats_and_fence():
    """step_async returns after the sync part; the mapper thread's work is visible in the stats and
    the next call waits for it.  With a compute stream registered, unmaps wait on the fence."""
    L = 8
    va.init_kvcache(L, 8, 128, 8, 32768, 0, torch.bfloat16, 2 * MB, False)
    va.reserve_physical_pages(2048 * MB)
    va.set_compute_stream(torch.cuda.current_stream().cuda_stream, True)
    tpp = va.get_config()["tokens_per_page"]
    lens = [tpp - 1] * 4 + [0] * 4
    va.step_async(lens)            # prefill arrivals: 4 blocks mapped on the critical path
    s0 = va.get_step_stats()
    assert s0["sync_pages_mapped"] == 4 * 2 * L
    # look-ahead (+2..+9 tokens) crosses into page 2, but the pass stops after
    # EAGER_NUM_KVBLOCKS = 2 blocks (vattention.cu:487,520-524)
    assert s0["async_pages_mapped"] == 2 * 2 * L
    lens = [tpp] * 4 + [0] * 4
    va.step_async(lens)            # nothing left to do synchronously: pages were pre-mapped
    s1 = va.get_step_stats()
    assert s1["sync_pages_mapped"] == 0
    assert s1["critical_path_ns"] < s0["critical_path_ns"]
    va.step([0] * 8, True)          # eager reclaim: unmap everything behind the fence
    assert va.get_state()["mapped_pages"] == [0] * 8


def test_megacache_tensor_core_path_respects_unmapped_pages():
    """Megacache views have a row pitch of L*Hkv*D*2 bytes (here 32 KB -> 64 tokens per 2 MB page),
    so a 128-row TMA box would run past a request's mapped prefix.  The tensor-core kernels fetch
    the last tile in 64-row boxes instead; this test would die with an illegal address otherwise.
    Decode (append) and chunked prefill both read straight from the virtual tensors."""
    L, Hkv, D, Hq, B, ctx = 32, 4, 128, 16, 4, 8192
    dtype = torch.bfloat16
    k_mega, v_mega = va.init_kvcache(L, Hkv, D, B, ctx, 0, dtype, 2 * MB, True)
    assert va.get_config()["tokens_per_page"] == 64
    va.reserve_physical_pages(512 * MB)
    lens_now = [700, 0, 130, 65]
    va.step(lens_now, True)
    assert va.get_state()["mapped_pages"] == [11, 0, 3, 2]
    layer = 5
    kc, vc = k_mega[:, :, layer], v_mega[:, :, layer]
    g = torch.Generator().manual_seed(5)
    host = {}
    for r, n in enumerate(lens_now):
        if n:
            k = torch.randn(n, Hkv, D, generator=g).to(dtype)
            v = torch.randn(n, Hkv, D, generator=g).to(dtype)
            host[r] = (k, v)
            att.cache_flat(k.cuda(), v.cuda(), kc[r], vc[r], "auto")
    # decode: one new token per active sequence; lengths grow by one (still inside the mapped pages)
    rids = [0, 2, 3]
    va.step([n + 1 if n else 0 for n in lens_now], True)
    q = torch.randn(3, 1, Hq, D, generator=g).to(dtype)
    kn = torch.randn(3, 1, Hkv, D, generator=g).to(dtype)
    vn = torch.randn(3, 1, Hkv, D, generator=g).to(dtype)
    seqlens = torch.tensor([lens_now[r] for r in rids], dtype=torch.int32)
    idx = torch.tensor(rids, dtype=torch.int32)
    max_len = max(lens_now) + 1
    out = att.flash_attn_with_kvcache(q.cuda(), kc[:, :max_len], vc[:, :max_len], kn.cuda(), vn.cuda(),
                                      cache_seqlens=seqlens.cuda(), cache_batch_idx=idx.cuda(), causal=True,
                                      impl="tc")
    torch.cuda.synchronize()
    kref = torch.zeros(B, max_len, Hkv, D, dtype=dtype)
    vref = torch.zeros(B, max_len, Hkv, D, dtype=dtype)
    for r, (k, v) in host.items():
        kref[r, :k.shape[0]], vref[r, :k.shape[0]] = k, v
    want = ref.attn_with_kvcache_ref(q, kref, vref, kn, vn, seqlens, idx, causal=True)
    scale = want.float().abs().max().item()
    assert (out.float().cpu() - want.float()).abs().max().item() <= 3e-3 * scale + 2 ** -7 * scale
    # chunked prefill of request 0: 96 new queries over its 701 cached tokens (total stays 701)
    qp = torch.randn(1, 96, Hq, D, generator=g).to(dtype)
    total = torch.tensor([701], dtype=torch.int32)
    outp = att.flash_attn_with_kvcache(qp.cuda(), kc[0:1], vc[0:1], cache_seqlens=total.cuda(), causal=True,
                                       impl="tc")
    torch.cuda.synchronize()
    wantp = ref.attn_with_kvcache_ref(qp, kref[0:1], vref[0:1], cache_seqlens=total, causal=True)
    scale = wantp.float().abs().max().item()
    assert (outp.float().cpu() - wantp.float()).abs().max().item() <= 3e-3 * scale + 2 ** -7 * scale


def test_map_common_pages_alias_on_the_real_driver():
    """Prefix sharing (vattention.cu:325-373, mux.h:68-85): after map_common_pages the SAME physical
    page backs the first blocks of every request -- bytes written through request 0's view are read
    back through request 1's and 2's; attention over either view gives the same result; physical
    memory is charged once; unmapping returns every page exactly once (oracle: ref-counted pool)."""
    L, Hkv, D, B, ctx = 2, 8, 128, 3, 8192
    ts = va.init_kvcache(L, Hkv, D, B, ctx, 0, torch.bfloat16, 2 * MB, False)
    n_pages = va.reserve_physical_pages(48 * MB)
    tpp = va.get_config()["tokens_per_page"]
    va.map_common_pages(tpp + 1)                     # 2 blocks shared by all 3 requests
    st = va.get_state()
    assert st["mapped_pages"] == [2, 2, 2]
    assert len(st["pool"]) == n_pages - 2 * 2 * L    # 2 blocks x (K, V) x L layers -- not x 3 requests
    g = torch.Generator(device="cuda").manual_seed(0)
    n = 2 * tpp
    for t in ts:
        t[0, :n].normal_(generator=g)                # write through request 0's virtual range only
    torch.cuda.synchronize()
    for t in ts:
        assert torch.equal(t[1, :n], t[0, :n]) and torch.equal(t[2, :n], t[0, :n])
    # a write through request 2 is seen by request 0 as well (aliases, not copies)
    ts[0][2, 5].fill_(3.0)
    torch.cuda.synchronize()
    assert torch.equal(ts[0][0, 5], torch.full_like(ts[0][0, 5], 3.0))
    # decode attention over the shared prefix: three requests, one physical copy
    q = torch.randn(1, 1, 32, D, device="cuda", generator=g).bfloat16().expand(B, 1, 32, D).contiguous()
    lens = torch.full((B,), n, dtype=torch.int32, device="cuda")
    out = att.flash_attn_with_kvcache(q, ts[0][:, :n], ts[L][:, :n], cache_seqlens=lens, causal=True)
    torch.cuda.synchronize()
    assert torch.equal(out[0], out[1]) and torch.equal(out[0], out[2])   # same bytes, same schedule, same bits
    want = ref.attn_with_kvcache_ref(q[:1].cpu(), ts[0][:1, :n].cpu(), ts[L][:1, :n].cpu(),
                                     cache_seqlens=lens[:1].cpu(), causal=True)
    err = (out[:1].float().cpu() - want.float()).abs().max().item()
    assert err <= 3e-3 * want.float().abs().max().item() + 1e-3
    # private growth on top of the shared prefix stays private
    va.step([n + 5, n, n], True)
    ts[0][0, n:n + 5].fill_(7.0)
    torch.cuda.synchronize()
    assert va.get_state()["mapped_pages"] == [3, 2, 2]
    va.step([0, 0, 0], True)                         # eager reclaim unmaps everything
    st = va.get_state()
    assert st["mapped_pages"] == [0, 0, 0]
    assert sorted(st["pool"]) == list(range(n_pages))   # every page back exactly once
