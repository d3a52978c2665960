"""ctypes binding of ``csrc/libmsegpu.so`` (C ABI: ``include/mse_b200.h``).

There is deliberately no CPU fallback: if the shared library is missing, or no sm_100a device
is present, the compute entry points raise ``NativeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import sys
from typing import Optional, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.environ.get("MSE_B200_LIB") or os.path.join(CSRC, "libmsegpu.so")   # override: experiments only
HEADER = os.path.join(os.path.dirname(HERE), "include", "mse_b200.h")

MSE_HOST, MSE_DEVICE, MSE_DEVICE_BORROW, MSE_HOST_ASYNC = 0, 1, 2, 3
STATUS_WORDS = 4
COMM_ID_BYTES = 128
MAX_TOPK = 4096
EMB_DIM = 768
KERNELS = {"bm25_score": 0, "topk_select": 1, "dense_scan": 2, "rerank": 3, "bm25_prepare": 4, "exchange": 5}

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


class NativeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"mse_b200 error {code}: {msg}")
        self.code = code


def build(verbose: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    src = os.path.join(CSRC, "api.cu")
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))] + [HEADER]
    if os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or \
        os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")      # a shell without the toolkit on PATH
    extra = os.environ.get("MSE_NVCC_FLAGS", "").split()          # experiments, e.g. -DMSE_BM25_RANGE16=4096
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, src]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB_PATH


_lib = None

_i32p, _f32p, _i64p, _vp = C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_int64), C.c_void_p

_SIGNATURES = {
    "mse_last_error": (C.c_char_p, []),
    "mse_abi_version": (C.c_int, []),
    "mse_device_count": (C.c_int, [_i32p]),
    "mse_index_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "mse_index_destroy": (C.c_int, [_vp]),
    "mse_index_set_option": (C.c_int, [_vp, C.c_char_p, C.c_int64]),
    "mse_bm25_load": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp,
                                C.c_float, C.c_float, C.c_float, C.c_int]),
    "mse_bm25_search_batch": (C.c_int, [_vp, C.c_int32, _vp, _vp, _vp, C.c_int32, C.c_float, _vp, _vp, _vp, C.c_int, _vp]),
    "mse_bm25_search_batch_async": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, _vp, C.c_int32, C.c_float, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "mse_bm25_last_stats": (C.c_int, [_vp, _i64p]),
    "mse_bm25_aggregate": (C.c_int, [C.c_int, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _i64p, C.c_int, _vp]),
    "mse_kernel_time": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double), _i64p]),
    "mse_dense_load": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_int, _vp, C.c_int]),
    "mse_dense_scan_batch": (C.c_int, [_vp, C.c_int32, _vp, C.c_int32, _vp, _vp, _vp, C.c_int, _vp]),
    "mse_dense_set_url_groups": (C.c_int, [_vp, _vp, C.c_int64, C.c_int]),
    "mse_dense_scan_batch_async": (C.c_int, [_vp, C.c_int32, _vp, C.c_int32, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "mse_hybrid_search_batch": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, C.c_int32, C.c_float, C.c_float, C.c_int32, C.c_int32,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "mse_comm_unique_id": (C.c_int, [_vp]),
    "mse_comm_init": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32]),
    "mse_comm_attach": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32]),
    "mse_comm_destroy": (C.c_int, [_vp]),
    "mse_bm25_search_sharded": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, _vp, C.c_int32, C.c_float, C.c_int32, _vp, _vp, _vp, _vp, _vp]),
    "mse_hybrid_search_sharded": (C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, C.c_int32, C.c_float, C.c_int32, C.c_float,
                                            C.c_int32, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mse_dense_scan_sharded": (C.c_int, [_vp, C.c_int32, _vp, C.c_int32, _vp, _vp, _vp, _vp, _vp]),
    "mse_rerank_batch": (C.c_int, [_vp, C.c_int32, _vp, _vp, _vp, _vp, _vp, C.c_float, C.c_int32, C.c_int32,
                                   _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "mse_rerank_shard_cos": (C.c_int, [_vp, C.c_int32, _vp, _vp, _vp, _vp, C.c_int64, _vp, C.c_int32,
                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mse_rerank_shard_fuse": (C.c_int, [_vp, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, C.c_int32,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mse_topk_merge": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp, C.c_int, _vp]),
}


def exported_symbols():
    return sorted(_SIGNATURES)


def lib():
    """Loads the shared library; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(-1, f"{LIB_PATH} is missing — run `python -c 'import __graft_entry__ as g; g.build()'`; "
                                  "this package has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise NativeError(rc, lib().mse_last_error().decode("utf-8", "replace"))


def device_count() -> int:
    n = C.c_int32(0)
    rc = lib().mse_device_count(C.byref(n))
    return 0 if rc else int(n.value)


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _ptr(x, dtype, where: int):
    """Address of a contiguous numpy array (host) or torch tensor (host or device) of `dtype`."""
    if x is None:
        return None
    if _is_torch(x):
        import torch
        want = {np.int32: torch.int32, np.int64: torch.int64, np.float32: torch.float32,
                "bf16": torch.bfloat16}[dtype]
        assert x.dtype == want, (x.dtype, want)
        assert x.is_contiguous()
        assert x.is_cuda == (where == MSE_DEVICE), "buffer location does not match `where`"
        assert where != MSE_HOST_ASYNC or x.is_pinned(), "MSE_HOST_ASYNC needs pinned host buffers"
        return C.c_void_p(x.data_ptr())
    assert where == MSE_HOST, "numpy buffers are (pageable) host memory"
    assert x.dtype == np.dtype(dtype) and x.flags["C_CONTIGUOUS"], (x.dtype, dtype)
    return C.c_void_p(x.ctypes.data)


def _where_of(*xs) -> int:
    for x in xs:
        if x is not None and _is_torch(x) and x.is_cuda:
            return MSE_DEVICE
    return MSE_HOST


def _stream_ptr(where: int, stream=None):
    """cudaStream_t of the call: an explicit torch stream / raw handle, else torch's current stream for device and
    pinned-async buffers, else the default stream."""
    if stream is not None:
        return C.c_void_p(int(getattr(stream, "cuda_stream", stream)))
    if where in (MSE_DEVICE, MSE_HOST_ASYNC):
        import torch
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)
    return None


def comm_unique_id() -> bytes:
    """NCCL unique id (create on rank 0, hand to every rank, pass to ``NativeIndex.comm_init``)."""
    buf = C.create_string_buffer(COMM_ID_BYTES)
    _check(lib().mse_comm_unique_id(buf))
    return bytes(buf.raw)


def bm25_aggregate(doc_tok_off, tok_term, n_terms: int, device: int = 0):
    """Device aggregation of tokenised documents (CSR of term ids) into the CSR posting arrays of the BM25 index
    (``mse_bm25_aggregate``).  Host arrays in, host arrays out: (term_off int64[V+1], post_doc int32[P], post_tf int32[P],
    total_freq int64[V])."""
    doc_tok_off = np.ascontiguousarray(doc_tok_off, dtype=np.int64)
    tok_term = np.ascontiguousarray(tok_term, dtype=np.int32)
    n_docs, T = int(doc_tok_off.shape[0]) - 1, int(tok_term.shape[0])
    term_off = np.empty(n_terms + 1, np.int64)
    post_doc, post_tf = np.empty(max(T, 1), np.int32), np.empty(max(T, 1), np.int32)
    total_freq = np.empty(max(n_terms, 1), np.int64)
    n_post = C.c_int64(0)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _check(lib().mse_bm25_aggregate(int(device), n_docs, int(n_terms), vp(doc_tok_off), vp(tok_term), vp(term_off), vp(post_doc),
                                    vp(post_tf), vp(total_freq), C.byref(n_post), MSE_HOST, None))
    P = int(n_post.value)
    return term_off, post_doc[:P].copy(), post_tf[:P].copy(), total_freq[:n_terms]


class NativeIndex:
    """Owns one ``mse_index`` (all device memory of one shard on one GPU)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(lib().mse_index_create(int(device), C.byref(self._h)))
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().mse_index_destroy(self._h)
            self._h = C.c_void_p()
        self._borrowed = None                            # a closed index no longer reads the tensor lent by dense_load

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name: str, value: int):
        _check(lib().mse_index_set_option(self._h, name.encode(), int(value)))

    def kernel_time(self, kernel: str) -> Tuple[float, int]:
        ms, n = C.c_double(0), C.c_int64(0)
        _check(lib().mse_kernel_time(self._h, KERNELS[kernel], C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def bm25_stats(self) -> dict:
        arr = (C.c_int64 * 8)()
        _check(lib().mse_bm25_last_stats(self._h, arr))
        return {"postings": arr[0], "emitted": arr[1], "rerun_queries": arr[2], "ranges": arr[3], "ctas": arr[4],
                "postings_looked_up": arr[5], "exact_mode_tasks": arr[6]}

    # ---- BM25 --------------------------------------------------------------------------------
    def bm25_load(self, term_off, post_doc, post_tf, doc_len, idf, avgdl, k1=1.2, b=0.75, doc_base=0):
        where = _where_of(term_off, post_doc, post_tf, doc_len, idf)
        n_terms, n_docs = int(term_off.shape[0]) - 1, int(doc_len.shape[0])
        _check(lib().mse_bm25_load(self._h, n_terms, n_docs, int(doc_base), _ptr(term_off, np.int64, where),
                                   _ptr(post_doc, np.int32, where), _ptr(post_tf, np.int32, where),
                                   _ptr(doc_len, np.int32, where), _ptr(idf, np.float32, where),
                                   float(avgdl), float(k1), float(b), where))

    def bm25_search(self, q_off, q_term, q_tf, top_k: int, min_score: float = 0.0, out=None):
        where = _where_of(q_off, q_term, q_tf)
        B = int(q_off.shape[0]) - 1
        if out is None:
            if where == MSE_DEVICE:
                import torch
                dev = q_off.device
                out = (torch.empty((B, top_k), dtype=torch.int32, device=dev),
                       torch.empty((B, top_k), dtype=torch.float32, device=dev),
                       torch.empty((B,), dtype=torch.int32, device=dev))
            else:
                out = (np.empty((B, top_k), np.int32), np.empty((B, top_k), np.float32), np.empty((B,), np.int32))
        o_doc, o_score, o_count = out
        _check(lib().mse_bm25_search_batch(self._h, B, _ptr(q_off, np.int32, where), _ptr(q_term, np.int32, where),
                                           _ptr(q_tf, np.int32, where), int(top_k), float(min_score),
                                           _ptr(o_doc, np.int32, where), _ptr(o_score, np.float32, where),
                                           _ptr(o_count, np.int32, where), where, _stream_ptr(where)))
        return out

    # ---- dense --------------------------------------------------------------------------------
    def dense_load(self, emb, doc_chunk_off, doc_base=0, chunk_base=0, borrow=False):
        """``borrow=True`` (bf16 CUDA tensor only): the index scans the tensor in place instead of copying it
        (a 77-154 GB shard cannot be resident twice); the tensor is kept alive by this object."""
        where = _where_of(emb, doc_chunk_off)
        is_bf16 = _is_torch(emb) and str(emb.dtype) == "torch.bfloat16"
        n_chunks, n_docs = int(emb.shape[0]), int(doc_chunk_off.shape[0]) - 1
        assert emb.shape[1] == EMB_DIM
        flag = where
        if borrow:
            assert where == MSE_DEVICE and is_bf16, "borrow needs a bf16 CUDA tensor"
            flag = MSE_DEVICE_BORROW
        _check(lib().mse_dense_load(self._h, n_chunks, n_docs, int(doc_base), int(chunk_base),
                                    _ptr(emb, "bf16" if is_bf16 else np.float32, where), int(is_bf16),
                                    _ptr(doc_chunk_off, np.int64, where), flag))
        self._borrowed = emb if borrow else None

    def dense_scan(self, q, top_k: int, out=None):
        where = _where_of(q)
        B = int(q.shape[0])
        if out is None:
            if where == MSE_DEVICE:
                import torch
                out = (torch.empty((B, top_k), dtype=torch.int32, device=q.device),
                       torch.empty((B, top_k), dtype=torch.float32, device=q.device),
                       torch.empty((B,), dtype=torch.int32, device=q.device))
            else:
                out = (np.empty((B, top_k), np.int32), np.empty((B, top_k), np.float32), np.empty((B,), np.int32))
        _check(lib().mse_dense_scan_batch(self._h, B, _ptr(q, np.float32, where), int(top_k),
                                          _ptr(out[0], np.int32, where), _ptr(out[1], np.float32, where),
                                          _ptr(out[2], np.int32, where), where, _stream_ptr(where)))
        return out

    def rerank(self, cand_off, cand_doc, cand_bm25, q, url_group=None, smoothing=0.15, max_chunks=10, max_out=1000):
        where = _where_of(cand_off, cand_doc, cand_bm25, q)
        B = int(cand_off.shape[0]) - 1
        if where == MSE_DEVICE:
            import torch
            dev = q.device
            mk = lambda dt: torch.empty((B, max_out), dtype=dt, device=dev)
            out = (mk(torch.int32), mk(torch.float32), mk(torch.float32), mk(torch.int64),
                   torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B,), dtype=torch.int32, device=dev))
        else:
            out = (np.empty((B, max_out), np.int32), np.empty((B, max_out), np.float32), np.empty((B, max_out), np.float32),
                   np.empty((B, max_out), np.int64), np.empty((B,), np.int32), np.empty((B,), np.int32))
        _check(lib().mse_rerank_batch(self._h, B, _ptr(cand_off, np.int32, where), _ptr(cand_doc, np.int32, where),
                                      _ptr(cand_bm25, np.float32, where), _ptr(url_group, np.int32, where),
                                      _ptr(q, np.float32, where), float(smoothing), int(max_chunks), int(max_out),
                                      _ptr(out[0], np.int32, where), _ptr(out[1], np.float32, where),
                                      _ptr(out[2], np.float32, where), _ptr(out[3], np.int64, where),
                                      _ptr(out[4], np.int32, where), _ptr(out[5], np.int32, where),
                                      where, _stream_ptr(where)))
        return out

    MAX_CAND, MAX_CHUNKS = 1024, 10

    def rerank_shard_cos(self, cand_off, cand_doc, cand_bm25, q, n_docs_global: int, url_group=None, max_chunks=10):
        """Sharded rerank, step 1 (CUDA tensors only).  Returns the exchange arrays (cos, rows, chunk0) — to be
        summed over the ranks — and the replicated survivor description (surv_doc, surv_bm25, surv_count)."""
        import torch
        B, dev = int(cand_off.shape[0]) - 1, q.device
        cos = torch.empty((B, self.MAX_CAND, self.MAX_CHUNKS), dtype=torch.float32, device=dev)
        rows = torch.empty((B, self.MAX_CAND), dtype=torch.int32, device=dev)
        chunk0 = torch.empty((B, self.MAX_CAND), dtype=torch.int64, device=dev)
        surv_doc = torch.empty((B, self.MAX_CAND), dtype=torch.int32, device=dev)
        surv_bm25 = torch.empty((B, self.MAX_CAND), dtype=torch.float32, device=dev)
        surv_count = torch.empty((B,), dtype=torch.int32, device=dev)
        D = MSE_DEVICE
        _check(lib().mse_rerank_shard_cos(self._h, B, _ptr(cand_off, np.int32, D), _ptr(cand_doc, np.int32, D),
                                          _ptr(cand_bm25, np.float32, D), _ptr(url_group, np.int32, D), int(n_docs_global),
                                          _ptr(q, np.float32, D), int(max_chunks), _ptr(cos, np.float32, D), _ptr(rows, np.int32, D),
                                          _ptr(chunk0, np.int64, D), _ptr(surv_doc, np.int32, D), _ptr(surv_bm25, np.float32, D),
                                          _ptr(surv_count, np.int32, D), _stream_ptr(D)))
        return (cos, rows, chunk0), (surv_doc, surv_bm25, surv_count)

    def rerank_shard_fuse(self, exchange, survivors, smoothing=0.15, max_out=1000):
        """Sharded rerank, step 2: outputs as ``rerank``."""
        import torch
        cos, rows, chunk0 = exchange
        surv_doc, surv_bm25, surv_count = survivors
        B, dev = int(cos.shape[0]), cos.device
        mk = lambda dt: torch.empty((B, max_out), dtype=dt, device=dev)
        out = (mk(torch.int32), mk(torch.float32), mk(torch.float32), mk(torch.int64),
               torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B,), dtype=torch.int32, device=dev))
        D = MSE_DEVICE
        _check(lib().mse_rerank_shard_fuse(self._h, B, _ptr(cos, np.float32, D), _ptr(rows, np.int32, D), _ptr(chunk0, np.int64, D),
                                           _ptr(surv_doc, np.int32, D), _ptr(surv_bm25, np.float32, D), _ptr(surv_count, np.int32, D),
                                           float(smoothing), int(max_out), _ptr(out[0], np.int32, D), _ptr(out[1], np.float32, D),
                                           _ptr(out[2], np.float32, D), _ptr(out[3], np.int64, D), _ptr(out[4], np.int32, D),
                                           _ptr(out[5], np.int32, D), _stream_ptr(D)))
        return out

    # ---- enqueue-only calls (MSE_DEVICE tensors or pinned host tensors) -----------------------------------------
    def new_status(self, like):
        """int32[4] status record in the memory space of `like` (a CUDA tensor or a pinned host tensor)."""
        import torch
        if like.is_cuda:
            return torch.zeros(STATUS_WORDS, dtype=torch.int32, device=like.device)
        return torch.zeros(STATUS_WORDS, dtype=torch.int32).pin_memory()

    def bm25_search_async(self, q_off, q_term, q_tf, n_slots: int, top_k: int, min_score: float = 0.0, out=None, status=None,
                          stream=None):
        """Enqueue-only BM25 (``mse_bm25_search_batch_async``): CUDA tensors (MSE_DEVICE) or pinned host tensors
        (MSE_HOST_ASYNC); results are valid in stream order / after the stream is synchronised."""
        import torch
        where = MSE_DEVICE if q_off.is_cuda else MSE_HOST_ASYNC
        B = int(q_off.shape[0]) - 1
        if out is None:
            mk = (lambda shape, dt: torch.empty(shape, dtype=dt, device=q_off.device)) if q_off.is_cuda else \
                (lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory())
            out = (mk((B, top_k), torch.int32), mk((B, top_k), torch.float32), mk((B,), torch.int32))
        _check(lib().mse_bm25_search_batch_async(self._h, B, int(n_slots), _ptr(q_off, np.int32, where), _ptr(q_term, np.int32, where),
                                                 _ptr(q_tf, np.int32, where), int(top_k), float(min_score),
                                                 _ptr(out[0], np.int32, where), _ptr(out[1], np.float32, where),
                                                 _ptr(out[2], np.int32, where), _ptr(status, np.int32, where), where,
                                                 _stream_ptr(where, stream)))
        return out

    def dense_scan_async(self, q, top_k: int, out=None, status=None, stream=None):
        import torch
        where = MSE_DEVICE if q.is_cuda else MSE_HOST_ASYNC
        B = int(q.shape[0])
        if out is None:
            mk = (lambda shape, dt: torch.empty(shape, dtype=dt, device=q.device)) if q.is_cuda else \
                (lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory())
            out = (mk((B, top_k), torch.int32), mk((B, top_k), torch.float32), mk((B,), torch.int32))
        _check(lib().mse_dense_scan_batch_async(self._h, B, _ptr(q, np.float32, where), int(top_k), _ptr(out[0], np.int32, where),
                                                _ptr(out[1], np.float32, where), _ptr(out[2], np.int32, where),
                                                _ptr(status, np.int32, where), where, _stream_ptr(where, stream)))
        return out

    def set_url_groups(self, url_group):
        """Stores the GLOBAL url-group ids (int32 per doc) in the index; rerank / hybrid calls use them by default."""
        if url_group is None:
            _check(lib().mse_dense_set_url_groups(self._h, None, 0, MSE_HOST))
            return
        where = _where_of(url_group)
        _check(lib().mse_dense_set_url_groups(self._h, _ptr(url_group, np.int32, where), int(url_group.shape[0]), where))

    @staticmethod
    def _rerank_out(B, max_out, like=None, pinned=False):
        if like is not None and _is_torch(like):
            import torch
            if like.is_cuda:
                mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=like.device)
            elif pinned:
                mk = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
            else:
                mk = lambda shape, dt: torch.empty(shape, dtype=dt)
            return (mk((B, max_out), torch.int32), mk((B, max_out), torch.float32), mk((B, max_out), torch.float32),
                    mk((B, max_out), torch.int64), mk((B,), torch.int32), mk((B,), torch.int32))
        return (np.empty((B, max_out), np.int32), np.empty((B, max_out), np.float32), np.empty((B, max_out), np.float32),
                np.empty((B, max_out), np.int64), np.empty((B,), np.int32), np.empty((B,), np.int32))

    def hybrid_search(self, q_off, q_term, q_tf, q_vec, top_k: int = 1000, min_score: float = 0.0, smoothing=0.15, max_chunks=10,
                      max_out=100, n_slots: Optional[int] = None, out=None, status=None, stream=None, pinned_async: bool = False):
        """BM25 top_k -> rerank -> max_out per query in ONE call (``mse_hybrid_search_batch``).  numpy / pageable torch:
        MSE_HOST (exact, complete on return); CUDA tensors: MSE_DEVICE (enqueue-only); pinned host tensors with
        ``pinned_async=True``: MSE_HOST_ASYNC.  ``n_slots`` = q_off[-1] (read here when the offsets are host memory)."""
        where = _where_of(q_off, q_term, q_tf, q_vec)
        if where == MSE_HOST and pinned_async:
            where = MSE_HOST_ASYNC
        B = int(q_off.shape[0]) - 1
        if n_slots is None:
            assert where != MSE_DEVICE, "pass n_slots with device-resident queries (no read-back in an enqueue-only call)"
            n_slots = int(q_off[-1])
        if out is None:
            out = self._rerank_out(B, max_out, q_off if _is_torch(q_off) else None, pinned=where == MSE_HOST_ASYNC)
        _check(lib().mse_hybrid_search_batch(self._h, B, int(n_slots), _ptr(q_off, np.int32, where), _ptr(q_term, np.int32, where),
                                             _ptr(q_tf, np.int32, where), _ptr(q_vec, np.float32, where), int(top_k), float(min_score),
                                             float(smoothing), int(max_chunks), int(max_out),
                                             _ptr(out[0], np.int32, where), _ptr(out[1], np.float32, where), _ptr(out[2], np.float32, where),
                                             _ptr(out[3], np.int64, where), _ptr(out[4], np.int32, where), _ptr(out[5], np.int32, where),
                                             _ptr(status, np.int32, where), where, _stream_ptr(where, stream)))
        return out

    # ---- corpus sharded by doc range over the GPUs of one box (NCCL inside the library) -------------------------------
    def comm_init(self, id_bytes: Optional[bytes], rank: int, world: int):
        buf = C.create_string_buffer(id_bytes, COMM_ID_BYTES) if id_bytes is not None else None
        _check(lib().mse_comm_init(self._h, buf, int(rank), int(world)))
        self.rank, self.world = int(rank), int(world)

    def comm_destroy(self):
        _check(lib().mse_comm_destroy(self._h))

    def bm25_search_sharded(self, q_off, q_term, q_tf, n_slots: int, top_k: int, min_score: float = 0.0, shard_list_len: int = 0,
                            out=None, status=None, stream=None):
        """The whole replicated batch in, this rank's block of the results out ([B/world, top_k])."""
        import torch
        D = MSE_DEVICE
        B = int(q_off.shape[0]) - 1
        bq = B // self.world
        if out is None:
            dev = q_off.device
            out = (torch.empty((bq, top_k), dtype=torch.int32, device=dev), torch.empty((bq, top_k), dtype=torch.float32, device=dev),
                   torch.empty((bq,), dtype=torch.int32, device=dev))
        _check(lib().mse_bm25_search_sharded(self._h, B, int(n_slots), _ptr(q_off, np.int32, D), _ptr(q_term, np.int32, D),
                                             _ptr(q_tf, np.int32, D), int(top_k), float(min_score), int(shard_list_len),
                                             _ptr(out[0], np.int32, D), _ptr(out[1], np.float32, D), _ptr(out[2], np.int32, D),
                                             _ptr(status, np.int32, D), _stream_ptr(D, stream)))
        return out

    def hybrid_search_sharded(self, q_off, q_term, q_tf, q_vec, n_slots: int, top_k: int = 1000, min_score: float = 0.0,
                              shard_list_len: int = 0, smoothing=0.15, max_chunks=10, max_out=100, out=None, status=None, stream=None):
        D = MSE_DEVICE
        B = int(q_off.shape[0]) - 1
        bq = B // self.world
        if out is None:
            out = self._rerank_out(bq, max_out, q_off)
        _check(lib().mse_hybrid_search_sharded(self._h, B, int(n_slots), _ptr(q_off, np.int32, D), _ptr(q_term, np.int32, D),
                                               _ptr(q_tf, np.int32, D), _ptr(q_vec, np.float32, D), int(top_k), float(min_score),
                                               int(shard_list_len), float(smoothing), int(max_chunks), int(max_out),
                                               _ptr(out[0], np.int32, D), _ptr(out[1], np.float32, D), _ptr(out[2], np.float32, D),
                                               _ptr(out[3], np.int64, D), _ptr(out[4], np.int32, D), _ptr(out[5], np.int32, D),
                                               _ptr(status, np.int32, D), _stream_ptr(D, stream)))
        return out

    def dense_scan_sharded(self, q, top_k: int, out=None, status=None, stream=None):
        import torch
        D = MSE_DEVICE
        B = int(q.shape[0])
        if out is None:
            out = (torch.empty((B, top_k), dtype=torch.int32, device=q.device), torch.empty((B, top_k), dtype=torch.float32, device=q.device),
                   torch.empty((B,), dtype=torch.int32, device=q.device))
        _check(lib().mse_dense_scan_sharded(self._h, B, _ptr(q, np.float32, D), int(top_k), _ptr(out[0], np.int32, D),
                                            _ptr(out[1], np.float32, D), _ptr(out[2], np.int32, D), _ptr(status, np.int32, D),
                                            _stream_ptr(D, stream)))
        return out

    def topk_merge(self, in_doc, in_score, in_count, top_k: int):
        """in_doc/in_score: [n_lists, B, list_k]; in_count: [n_lists, B]."""
        where = _where_of(in_doc, in_score, in_count)
        n_lists, B, list_k = (int(s) for s in in_doc.shape)
        if where == MSE_DEVICE:
            import torch
            dev = in_doc.device
            out = (torch.empty((B, top_k), dtype=torch.int32, device=dev), torch.empty((B, top_k), dtype=torch.float32, device=dev),
                   torch.empty((B,), dtype=torch.int32, device=dev))
        else:
            out = (np.empty((B, top_k), np.int32), np.empty((B, top_k), np.float32), np.empty((B,), np.int32))
        _check(lib().mse_topk_merge(self._h, B, n_lists, list_k, _ptr(in_doc, np.int32, where), _ptr(in_score, np.float32, where),
                                    _ptr(in_count, np.int32, where), int(top_k), _ptr(out[0], np.int32, where),
                                    _ptr(out[1], np.float32, where), _ptr(out[2], np.int32, where), where, _stream_ptr(where)))
        return out
