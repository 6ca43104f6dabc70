"""Replay an allocator API trace on the REFERENCE extension (oracle/_ref/vattention_ref*.so,
built unmodified from the original project's vattention/vattention.cu by oracle/Makefile) and dump
its state after every call as JSON.

TEST INFRASTRUCTURE ONLY.  Runs on the GPU box (the module needs libcuda).  State that the
reference does not expose through its API is read straight from its file-scope globals
(utils.h:22-69): they are non-static, so `mapped_pages`, `curr_seq_lengths`, `cuda_pages`
and `mem_manager_running` are exported data symbols; a std::vector<u64> is three pointers.
Physical handles are translated to their 0-based creation index (the pool right after
reserve_cuda_pages is in creation order, cudaInternal.h:51-56).

usage: python oracle/ref_driver.py trace.json out.json
trace: [["init", L, Hkv, D, B, ctx, "bf16"|"fp16", page, mega], ["reserve", bytes],
        ["step", lens, eager], ["step_async", lens], ["alloc", seqlen], ["free", reqId],
        ["nfree"], ["set_deferred", bool]]
"""
from __future__ import annotations

import ctypes
import glob
import importlib.util
import json
import os
import sys
import time


def load_ref():
    here = os.path.dirname(os.path.abspath(__file__))
    cands = glob.glob(os.path.join(here, "_ref", "vattention_ref*.so"))
    if not cands:
        raise SystemExit("oracle/_ref/vattention_ref*.so not built (run `make -C oracle REF=<checkout>/vattention`)")
    import torch  # noqa: F401  (libtorch must be loaded first)
    spec = importlib.util.spec_from_file_location("vattention_ref", cands[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, ctypes.CDLL(cands[0])


def read_vec_u64(dll, name):
    raw = (ctypes.c_void_p * 3).in_dll(dll, name)
    begin, end = raw[0] or 0, raw[1] or 0
    n = (end - begin) // 8
    if n == 0:
        return []
    return list((ctypes.c_uint64 * n).from_address(begin))


def wait_bg(dll):
    # the flag is raised inside the detached thread (vattention.cu:540-544): give it time to start
    flag = ctypes.c_bool.in_dll(dll, "mem_manager_running")
    time.sleep(0.02)
    while flag.value:
        time.sleep(0.001)
    time.sleep(0.005)
    while flag.value:
        time.sleep(0.001)


def main(trace_path, out_path):
    import torch
    torch.zeros(1, device="cuda")  # the reference needs torch's context to exist (cudaInternal.h:19-25)
    ref, dll = load_ref()
    trace = json.load(open(trace_path))
    handle_index = {}
    snaps = []
    for op in trace:
        ret, err = None, None
        try:
            if op[0] == "init":
                _, L, Hkv, D, B, ctx, dt, page, mega = op
                dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[dt]
                ts = ref.init_kvcache(L, Hkv, D, B, ctx, 0, dtype, page, bool(mega))
                ret = [len(ts), list(ts[0].shape), list(ts[0].stride())]
            elif op[0] == "reserve":
                ret = ref.reserve_physical_pages(op[1])
                for h in read_vec_u64(dll, "cuda_pages"):
                    if h not in handle_index:
                        handle_index[h] = len(handle_index)
            elif op[0] == "step":
                ref.step(op[1], bool(op[2]))
            elif op[0] == "step_async":
                ref.step_async(op[1])
                wait_bg(dll)
            elif op[0] == "alloc":
                ret = ref.alloc_new_batch_idx(op[1])
            elif op[0] == "free":
                ref.free_batch_idx(op[1])
            elif op[0] == "nfree":
                ret = ref.num_free_kvblocks()
            elif op[0] == "set_deferred":
                ref.set_deferred_reclamation(bool(op[1]))
            else:
                raise ValueError(op[0])
        except RuntimeError as e:
            err = str(e).splitlines()[0]
            ref.set_verbose(False)
        snaps.append({
            "op": op, "ret": ret, "err": err,
            "mapped_pages": read_vec_u64(dll, "mapped_pages"),
            "seq_lens": read_vec_u64(dll, "curr_seq_lengths"),
            "pool": [handle_index[h] for h in read_vec_u64(dll, "cuda_pages")],
            "num_free_kvblocks": ref.num_free_kvblocks() if op[0] != "init" or True else None,
        })
    json.dump(snaps, open(out_path, "w"))
    ref.cleanup()


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
