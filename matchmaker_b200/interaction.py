"""Torch-facing wrappers of the interaction kernels (C ABI in ``include/matchmaker_b200.h``).

PyTorch is plumbing here: it owns device memory and the current stream; the arithmetic runs in
``libmatchmaker_b200.so``.  No function in this module has a CPU or eager-PyTorch fallback.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib

_DTYPES = {torch.float16: _lib.F16, torch.bfloat16: _lib.BF16, torch.float32: _lib.F32}
_MASK_DTYPES = {torch.bool: _lib.MASK_U8, torch.uint8: _lib.MASK_U8, torch.int32: _lib.MASK_I32,
                torch.int64: _lib.MASK_I64, torch.float32: _lib.MASK_F32}
_IMPLS = {"auto": _lib.IMPL_AUTO, "simt": _lib.IMPL_SIMT, "tcgen05": _lib.IMPL_TCGEN05,
          "tcgen05_docm": _lib.IMPL_TCGEN05_DOCM, "tcgen05_ragged": _lib.IMPL_TCGEN05_RAGGED}


def _require_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.MatchmakerB200Error(
                "matchmaker_b200 interaction ops run on CUDA (sm_100a) tensors only; got a "
                f"{t.device} tensor and there is no CPU fallback")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise _lib.MatchmakerB200Error(f"tensors on different devices: {dev} vs {t.device}")
    return dev


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _prep_mask(m: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if m is None:
        return None
    if m.dtype not in _MASK_DTYPES:
        m = m != 0
    return m.contiguous()


def _common_mask_dtype(a: Optional[torch.Tensor], b: Optional[torch.Tensor]):
    """Both masks of one call share one element type (one `mask_dtype` argument)."""
    if a is not None and b is not None and a.dtype != b.dtype:
        a, b = (a != 0), (b != 0)
    code = _lib.MASK_NONE
    for m in (a, b):
        if m is not None:
            code = _MASK_DTYPES[m.dtype]
    return a, b, code


def maxsim(q: torch.Tensor, d: torch.Tensor, q_mask: Optional[torch.Tensor] = None,
           d_mask: Optional[torch.Tensor] = None, docs_per_query: int = 1,
           pair_q: Optional[torch.Tensor] = None, pair_d: Optional[torch.Tensor] = None,
           impl: str = "auto", return_argmax: bool = False, pair_dmask: Optional[torch.Tensor] = None):
    """ColBERT max-sim scores, fp32.

    q [n_q, Lq, dim], d [n_d, Ld, dim] (fp16 / bf16 / fp32, same dtype), masks [n, L] (nonzero =
    token).  Pair p scores query ``pair_q[p]`` (default ``p // docs_per_query``) against document
    ``pair_d[p]`` (default ``p``).  Semantics: matchmaker/models/colbert.py:68-75 / :100-112.

    Envelope: 1 <= Lq <= 128, 1 <= dim <= 1024, any Ld >= 1, with or without ``return_argmax``; ``impl="auto"``
    serves every such shape and raises :class:`MatchmakerB200Error` for any other.  ``impl="auto"`` picks the
    queries-on-M tcgen05 kernel (fp16/bf16, Lq <= 32, dim 64 or 128, 16-byte aligned q/d), else the
    documents-on-M tcgen05 kernel (fp16/bf16, dim % 64 == 0, no argmax, aligned, query tile small enough to
    leave room for two document stages in shared memory: e.g. Lq <= 32 at dim 768), else the SIMT kernel.
    A forced ``impl`` raises where its kernel does not cover the shape.
    """
    dev = _require_cuda(q, d, q_mask, d_mask, pair_q, pair_d, pair_dmask)
    if q.dtype != d.dtype or q.dtype not in _DTYPES:
        raise _lib.MatchmakerB200Error(f"q/d must share a dtype in fp16/bf16/fp32, got {q.dtype}, {d.dtype}")
    if q.dim() != 3 or d.dim() != 3 or q.shape[-1] != d.shape[-1]:
        raise _lib.MatchmakerB200Error(f"expected q [n_q,Lq,dim], d [n_d,Ld,dim]; got {tuple(q.shape)}, {tuple(d.shape)}")
    q = q.contiguous()
    d = d.contiguous()
    q_mask, d_mask, mcode = _common_mask_dtype(_prep_mask(q_mask), _prep_mask(d_mask))
    n_q, Lq, dim = q.shape
    n_d, Ld, _ = d.shape
    if q_mask is not None and tuple(q_mask.shape) != (n_q, Lq):
        raise _lib.MatchmakerB200Error("q_mask shape mismatch")
    if d_mask is not None and tuple(d_mask.shape) != (n_d, Ld):
        raise _lib.MatchmakerB200Error("d_mask shape mismatch")
    if pair_q is not None or pair_d is not None:
        if pair_q is None or pair_d is None:
            raise _lib.MatchmakerB200Error("pair_q and pair_d must be given together")
        pair_q = pair_q.to(torch.int32).contiguous()
        pair_d = pair_d.to(torch.int32).contiguous()
        n_pairs = pair_q.numel()
        if pair_d.numel() != n_pairs:
            raise _lib.MatchmakerB200Error("pair_q / pair_d length mismatch")
        if pair_dmask is not None:
            pair_dmask = pair_dmask.to(torch.int32).contiguous()
            if pair_dmask.numel() != n_pairs:
                raise _lib.MatchmakerB200Error("pair_dmask length mismatch")
    else:
        n_pairs = n_d
        if n_q * docs_per_query < n_d:
            raise _lib.MatchmakerB200Error("n_q * docs_per_query < n_d")
    out = torch.empty(n_pairs, dtype=torch.float32, device=dev)
    argmax = torch.empty((n_pairs, Lq), dtype=torch.int32, device=dev) if return_argmax else None
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_maxsim_fwd(_ptr(q), _ptr(d), _ptr(q_mask), _ptr(d_mask), _ptr(pair_q), _ptr(pair_d),
                                   _ptr(pair_dmask), _ptr(out), _ptr(argmax), n_q, n_d, n_pairs, docs_per_query, Lq, Ld, dim,
                                   _DTYPES[q.dtype], mcode, _IMPLS[impl], _stream(dev))
    _lib.check(rc, "mmb200_maxsim_fwd")
    return (out, argmax) if return_argmax else out


def maxsim_allpairs(q: torch.Tensor, q_mask: Optional[torch.Tensor], d: torch.Tensor,
                    d_mask: Optional[torch.Tensor], impl: str = "auto",
                    reference_mask_indexing: bool = False) -> torch.Tensor:
    """All query x document max-sim scores [n_q, n_d] (colbert.py:154-162).

    ``reference_mask_indexing=True`` reproduces the reference bit-for-bit: colbert.py:158 expands
    ``document_mask`` [n_d, Ld] along the *query* axis of the [n_q, n_d, Lq, Ld] score tensor, i.e. pair
    (a, b) is masked with the mask of document ``a`` (only defined for n_q == n_d, the in-batch case).
    The default applies each document's own mask."""
    n_q, n_d = q.shape[0], d.shape[0]
    idx = torch.arange(n_q * n_d, device=q.device, dtype=torch.int32)
    pq = torch.div(idx, n_d, rounding_mode="floor").to(torch.int32)
    pd = (idx - pq * n_d).to(torch.int32)
    pdm = None
    if reference_mask_indexing and d_mask is not None:
        if n_q != n_d:
            raise _lib.MatchmakerB200Error("reference mask indexing (colbert.py:158) needs n_q == n_d")
        pdm = pq
    return maxsim(q, d, q_mask, d_mask, pair_q=pq, pair_d=pd, impl=impl, pair_dmask=pdm).view(n_q, n_d)


def maxsim_bwd(q: torch.Tensor, d: torch.Tensor, grad_out: torch.Tensor, argmax: torch.Tensor,
               docs_per_query: int = 1) -> Tuple[torch.Tensor, torch.Tensor]:
    """Gradients of :func:`maxsim` (pairs mode) w.r.t. q and d, fp32."""
    dev = _require_cuda(q, d, grad_out, argmax)
    q = q.contiguous()
    d = d.contiguous()
    n_q, Lq, dim = q.shape
    n_d, Ld, _ = d.shape
    grad_out = grad_out.to(torch.float32).contiguous()
    gq = torch.empty((n_q, Lq, dim), dtype=torch.float32, device=dev)
    gd = torch.empty((n_d, Ld, dim), dtype=torch.float32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_maxsim_bwd(_ptr(q), _ptr(d), _ptr(grad_out), _ptr(argmax.contiguous()), _ptr(gq), _ptr(gd),
                                   n_q, n_d, n_d, docs_per_query, Lq, Ld, dim, _DTYPES[q.dtype], _stream(dev))
    _lib.check(rc, "mmb200_maxsim_bwd")
    return gq, gd


def maxsim_host(q: torch.Tensor, d: torch.Tensor, q_mask: Optional[torch.Tensor] = None,
                d_mask: Optional[torch.Tensor] = None, docs_per_query: int = 1, chunk_pairs: int = 0,
                device: Optional[torch.device] = None) -> torch.Tensor:
    """End-to-end max-sim over HOST tensors (pinned for full PCIe rate): document slabs are streamed to the
    GPU and scored while the next slab is in flight; returns a host fp32 tensor.  This is the call
    dense_retrieval.py:398-412 would make for token matrices gathered from the CPU memmap storage."""
    for t in (q, d, q_mask, d_mask):
        if t is not None and t.is_cuda:
            raise _lib.MatchmakerB200Error("maxsim_host takes host tensors; use maxsim() for device tensors")
    if q.dtype != d.dtype or q.dtype not in _DTYPES:
        raise _lib.MatchmakerB200Error("q/d must share a dtype in fp16/bf16/fp32")
    q = q.contiguous()
    d = d.contiguous()
    q_mask, d_mask, mcode = _common_mask_dtype(_prep_mask(q_mask), _prep_mask(d_mask))
    n_q, Lq, dim = q.shape
    n_d, Ld, _ = d.shape
    if n_q * docs_per_query < n_d:
        raise _lib.MatchmakerB200Error("n_q * docs_per_query < n_d")
    out = torch.empty(n_d, dtype=torch.float32, pin_memory=True)
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    with torch.cuda.device(dev):
        rc = lib.mmb200_maxsim_fwd_host(_ptr(q), _ptr(d), _ptr(q_mask), _ptr(d_mask), _ptr(out), n_q, n_d,
                                        docs_per_query, Lq, Ld, dim, _DTYPES[q.dtype], mcode, chunk_pairs)
    _lib.check(rc, "mmb200_maxsim_fwd_host")
    return out


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


def kernel_pool(q: torch.Tensor, d: torch.Tensor, q_mask: torch.Tensor, d_mask: torch.Tensor,
                mu: torch.Tensor, sigma: torch.Tensor, weight: torch.Tensor, alpha: Optional[torch.Tensor] = None,
                log_scale: float = 1.0, want_per_kernel: bool = False, want_per_kernel_query: bool = False,
                want_cosine: bool = False, impl: str = "auto", doc_gate: Optional[torch.Tensor] = None,
                clamp_min: float = 1e-10, bias: float = 0.0, save_for_backward: bool = False):
    """Cosine match matrix + RBF kernel pooling, forward (knrm.py:52-84 / ecai20_tk.py:105-124).

    q [B,Lq,D], d [B,Ld,D] fp32; masks [B,L]; mu/sigma/weight(/alpha) [K].  Returns a dict with "score"
    [B] and, on request, "per_kernel" [B,K], "per_kernel_query" [B,Lq,K], "cosine" [B,Lq,Ld].

    Variants: ``doc_gate`` [B,Ld] multiplies every activation of its document term (TK-Sparse,
    cikm20_tk_sparse.py:135); ``clamp_min`` / ``bias`` are the 1e-4 floor and the Linear bias of IDCM's ESM scorer
    (sigir21_idcm.py:185-186).

    ``save_for_backward=True`` (shapes for which :func:`kernel_pool_train_supported` holds) runs the
    training forward: the result additionally carries "saved", the opaque state the tensor-core backward consumes
    (:func:`kernel_pool_bwd` with ``saved=``), and "per_kernel_query"."""
    dev = _require_cuda(q, d, q_mask, d_mask, mu, sigma, weight, alpha, doc_gate)
    if q.dtype != torch.float32 or d.dtype != torch.float32:
        q, d = q.float(), d.float()  # the reference runs TK/KNRM with use_fp16: False (tk.yaml:6)
    q, d = q.contiguous(), d.contiguous()
    B, Lq, D = q.shape
    _, Ld, _ = d.shape
    if d.shape[0] != B or d.shape[2] != D:
        raise _lib.MatchmakerB200Error(f"shape mismatch: q {tuple(q.shape)} d {tuple(d.shape)}")
    q_mask, d_mask, mcode = _common_mask_dtype(_prep_mask(q_mask), _prep_mask(d_mask))
    mu, sigma, weight = _f32c(mu).view(-1), _f32c(sigma).view(-1), _f32c(weight).view(-1)
    alpha = None if alpha is None else _f32c(alpha).view(-1)
    K = mu.numel()
    score = torch.empty(B, dtype=torch.float32, device=dev)
    pk = torch.empty((B, K), dtype=torch.float32, device=dev) if want_per_kernel else None
    pkq = torch.empty((B, Lq, K), dtype=torch.float32, device=dev) if want_per_kernel_query else None
    cos = torch.empty((B, Lq, Ld), dtype=torch.float32, device=dev) if want_cosine else None
    gate = None
    if doc_gate is not None:
        gate = _f32c(doc_gate).reshape(B, Ld)
    lib = _lib.load()
    if save_for_backward:
        if want_cosine or not kernel_pool_train_supported(Lq, Ld, D, K):
            raise _lib.MatchmakerB200Error("kernel_pool(save_for_backward=True): outside the tensor-core training envelope")
        if pkq is None:
            pkq = torch.empty((B, Lq, K), dtype=torch.float32, device=dev)
        saved = torch.empty(int(lib.mmb200_kernel_pool_saved_floats(B, Ld)), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = lib.mmb200_kernel_pool_fwd_train(_ptr(q), _ptr(d), _ptr(q_mask), _ptr(d_mask), _ptr(gate), _ptr(mu), _ptr(sigma),
                                                  _ptr(alpha), _ptr(weight), _ptr(score), _ptr(pk), _ptr(pkq), _ptr(saved),
                                                  B, Lq, Ld, D, K, float(log_scale), float(clamp_min), float(bias), mcode,
                                                  _stream(dev))
        _lib.check(rc, "mmb200_kernel_pool_fwd_train")
        return {"score": score, "per_kernel": pk, "per_kernel_query": pkq, "cosine": None, "saved": saved}
    with torch.cuda.device(dev):
        rc = lib.mmb200_kernel_pool_fwd_ex(_ptr(q), _ptr(d), _ptr(q_mask), _ptr(d_mask), _ptr(gate), _ptr(mu), _ptr(sigma),
                                           _ptr(alpha), _ptr(weight), _ptr(score), _ptr(pk), _ptr(pkq), _ptr(cos),
                                           B, Lq, Ld, D, K, float(log_scale), float(clamp_min), float(bias), mcode,
                                           _IMPLS[impl], _stream(dev))
    _lib.check(rc, "mmb200_kernel_pool_fwd_ex")
    return {"score": score, "per_kernel": pk, "per_kernel_query": pkq, "cosine": cos}


def kernel_pool_train_supported(Lq: int, Ld: int, D: int, K: int) -> bool:
    """True when the tensor-core training pair (forward that saves its cosines + tcgen05 backward) covers the shape."""
    return bool(_lib.load().mmb200_kernel_pool_train_tc_supported(int(Lq), int(Ld), int(D), int(K)))


def kernel_pool_bwd(q, d, q_mask, d_mask, mu, sigma, weight, alpha, per_kernel_query, grad_score,
                    log_scale: float = 1.0, doc_gate: Optional[torch.Tensor] = None, clamp_min: float = 1e-10,
                    saved: Optional[torch.Tensor] = None):
    """Backward of :func:`kernel_pool`: returns (grad_q, grad_d, grad_alpha or None, grad_weight[, grad_gate when a
    ``doc_gate`` was given]).  With ``saved`` (from ``kernel_pool(save_for_backward=True)``) both contractions run on the
    tensor cores (tf32 operands: gradients within a few 1e-4 relative of the fp32 expression)."""
    dev = _require_cuda(q, d, per_kernel_query, grad_score)
    q, d = q.float().contiguous(), d.float().contiguous()
    B, Lq, D = q.shape
    Ld = d.shape[1]
    q_mask, d_mask, mcode = _common_mask_dtype(_prep_mask(q_mask), _prep_mask(d_mask))
    mu, sigma, weight = _f32c(mu).view(-1), _f32c(sigma).view(-1), _f32c(weight).view(-1)
    alpha_c = None if alpha is None else _f32c(alpha).view(-1)
    K = mu.numel()
    gq = torch.empty_like(q)
    gd = torch.empty_like(d)
    ga = torch.empty(K, dtype=torch.float32, device=dev)
    gw = torch.empty(K, dtype=torch.float32, device=dev)
    ws = torch.empty(2 * B * K, dtype=torch.float32, device=dev)
    gate = None if doc_gate is None else _f32c(doc_gate).reshape(B, Ld)
    gg = None if doc_gate is None else torch.empty((B, Ld), dtype=torch.float32, device=dev)
    lib = _lib.load()
    if saved is not None:
        with torch.cuda.device(dev):
            rc = lib.mmb200_kernel_pool_bwd_saved(_ptr(q), _ptr(d), _ptr(q_mask), _ptr(d_mask), _ptr(gate), _ptr(mu), _ptr(sigma),
                                                  _ptr(alpha_c), _ptr(weight), _ptr(per_kernel_query.contiguous()),
                                                  _ptr(saved), _ptr(_f32c(grad_score)), _ptr(gq), _ptr(gd), _ptr(gg), _ptr(ga),
                                                  _ptr(gw), _ptr(ws), B, Lq, Ld, D, K, float(log_scale), float(clamp_min),
                                                  mcode, _stream(dev))
        _lib.check(rc, "mmb200_kernel_pool_bwd_saved")
        if doc_gate is not None:
            return gq, gd, (ga if alpha is not None else None), gw, gg
        return gq, gd, (ga if alpha is not None else None), gw
    with torch.cuda.device(dev):
        rc = lib.mmb200_kernel_pool_bwd_ex(_ptr(q), _ptr(d), _ptr(q_mask), _ptr(d_mask), _ptr(gate), _ptr(mu), _ptr(sigma),
                                           _ptr(alpha_c), _ptr(weight), _ptr(per_kernel_query.contiguous()),
                                           _ptr(_f32c(grad_score)), _ptr(gq), _ptr(gd), _ptr(gg), _ptr(ga), _ptr(gw),
                                           _ptr(ws), B, Lq, Ld, D, K, float(log_scale), float(clamp_min), mcode,
                                           _stream(dev))
    _lib.check(rc, "mmb200_kernel_pool_bwd_ex")
    if doc_gate is not None:
        return gq, gd, (ga if alpha is not None else None), gw, gg
    return gq, gd, (ga if alpha is not None else None), gw


def dot_pairs(qv: torch.Tensor, dv: torch.Tensor) -> torch.Tensor:
    """score[b] = <qv[b], dv[b]> in fp32 (bert_dot.py:62).  qv, dv [B, dim], same dtype."""
    dev = _require_cuda(qv, dv)
    if qv.dtype != dv.dtype or qv.dtype not in _DTYPES or qv.shape != dv.shape or qv.dim() != 2:
        raise _lib.MatchmakerB200Error(f"dot_pairs expects two [B,dim] tensors of one dtype, got {tuple(qv.shape)} "
                                       f"{qv.dtype} / {tuple(dv.shape)} {dv.dtype}")
    qv, dv = qv.contiguous(), dv.contiguous()
    out = torch.empty(qv.shape[0], dtype=torch.float32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_dot_pairs(_ptr(qv), _ptr(dv), _ptr(out), qv.shape[0], qv.shape[1], _DTYPES[qv.dtype],
                                  _stream(dev))
    _lib.check(rc, "mmb200_dot_pairs")
    return out


TKL_CHUNK, TKL_WINDOW = 40, 30
_TKL_COVER_CACHE = {}


def tkl_kernel_set_covers(mu: torch.Tensor, sigma: torch.Tensor) -> bool:
    """True when every cosine in [-1, 1] activates at least one RBF kernel under ex2.approx.ftz, i.e. when the window
    token count of sigir20_tkl.py:210 equals the count of unmasked positions (tkl_ts.cu explains why that matters).
    Same sweep as the device-side plan kernel; evaluated on the host once per (mu, sigma) tensor version -- they are
    constant buffers of the model -- so that the launch path knows which kernel to enqueue without a device round trip."""
    key = (mu.data_ptr(), mu._version, sigma.data_ptr(), sigma._version, mu.numel())
    hit = _TKL_COVER_CACHE.get(key)
    if hit is not None:
        return hit
    m, sg = mu.detach().float().view(-1).cpu().tolist(), sigma.detach().float().view(-1).cpu().tolist()
    x, ok = -1.01, True
    while x < 1.01:
        reach = x
        for mk, sk in zip(m, sg):
            h = 11.0 * sk / (0.5 * 1.4426950408889634) ** 0.5
            if mk - h <= x and mk + h > reach:
                reach = mk + h
        if reach <= x:
            ok = False
            break
        x = reach
    if len(_TKL_COVER_CACHE) > 64:
        _TKL_COVER_CACHE.clear()
    _TKL_COVER_CACHE[key] = ok
    return ok


def tkl_window_scores(q_ctx: torch.Tensor, q_mask: torch.Tensor, doc_chunks: torch.Tensor, chunk_mask: torch.Tensor,
                      packed_indices: torch.Tensor, chunk_pieces: int, mu: torch.Tensor, sigma: torch.Tensor,
                      dense_weight: torch.Tensor, saturation: str, sat_params: torch.Tensor,
                      sat_red_weight: Optional[torch.Tensor] = None, impl: str = "auto") -> torch.Tensor:
    """Window scores [B, W] of the TKL interaction stage (sigir20_tkl.py:180-252).

    ``packed_indices`` [B*C] bool is the reference's chunk packing mask (:159); ``doc_chunks`` [Nc,40,D] /
    ``chunk_mask`` [Nc,40] are the packed, contextualised chunks without overlap (:174-175)."""
    dev = _require_cuda(q_ctx, q_mask, doc_chunks, chunk_mask, packed_indices, mu, sigma, dense_weight, sat_params)
    q_ctx = q_ctx.float().contiguous()
    doc_chunks = doc_chunks.float().contiguous()
    B, Lq, D = q_ctx.shape
    C = int(chunk_pieces)
    if packed_indices.numel() != B * C or doc_chunks.shape[1] != TKL_CHUNK:
        raise _lib.MatchmakerB200Error("tkl_window_scores: inconsistent chunk packing")
    slot_to_packed = _tkl_slot_map(packed_indices)
    q_mask, chunk_mask, mcode = _common_mask_dtype(_prep_mask(q_mask), _prep_mask(chunk_mask))
    mu, sigma, dense_weight = _f32c(mu).view(-1), _f32c(sigma).view(-1), _f32c(dense_weight).view(-1)
    sat_params = _f32c(sat_params).view(-1)
    sat_code = {"embedding": 0, "log": 1}[saturation]
    red = None if sat_red_weight is None else _f32c(sat_red_weight).view(-1)
    K = mu.numel()
    W = (C * TKL_CHUNK - TKL_WINDOW) // 2 + 1
    out = torch.empty((B, W), dtype=torch.float32, device=dev)
    if impl == "auto":
        # decide on the host (cached per parameter version) so that only ONE of the two kernels is enqueued; the library's
        # own device-side check stays in force (a forced tcgen05 call on a kernel set without cover writes zeros)
        impl = "tcgen05" if (Lq * K <= 512 and K <= 16 and tkl_kernel_set_covers(mu, sigma)) else "simt"
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_tkl_window_scores(_ptr(q_ctx), _ptr(q_mask), _ptr(doc_chunks), _ptr(chunk_mask),
                                          _ptr(slot_to_packed), _ptr(mu), _ptr(sigma), _ptr(dense_weight), _ptr(red),
                                          _ptr(sat_params), _ptr(out), B, doc_chunks.shape[0], Lq, D, C, K, sat_code, mcode,
                                          _IMPLS[impl], _stream(dev))
    _lib.check(rc, "mmb200_tkl_window_scores")
    return out


def tkl_top_hills(window_score: torch.Tensor, chunk_scoring: torch.Tensor):
    """Greedy top-3 windows with +-15 suppression, +-1/+-2 neighbours, weighted sum (sigir20_tkl.py:254-286).
    Returns (score [B], orig_score [B,W], top_idx [B,3] int64, top15 [B,15]); ``window_score`` is not modified."""
    dev = _require_cuda(window_score, chunk_scoring)
    ws = window_score.float().contiguous()
    B, W = ws.shape
    orig = torch.empty_like(ws)
    top_idx = torch.empty((B, 3), dtype=torch.int64, device=dev)
    top15 = torch.empty((B, 15), dtype=torch.float32, device=dev)
    score = torch.empty(B, dtype=torch.float32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_tkl_top_hills(_ptr(ws), _ptr(orig), _ptr(_f32c(chunk_scoring).view(-1)), _ptr(top_idx), _ptr(top15),
                                      _ptr(score), B, W, _stream(dev))
    _lib.check(rc, "mmb200_tkl_top_hills")
    return score, orig, top_idx, top15


FLAT_IP_MAX_K = 1024


def flat_ip_split_f32(x: torch.Tensor, role: str, scale_log2: Optional[int] = None) -> Tuple[torch.Tensor, int]:
    """fp32 vectors -> the fp16 hi / lo layout of MMB200_F32_SPLIT16: x * 2^s = hi + lo (+ a 2^-22 relative residue),
    s chosen so that the largest magnitude sits just below 2^15 (fp16 range, lo halves stay normal numbers).
    role "passages": [n, 2*dim] = [hi | lo] (the index stores this once); role "queries": [nq, 3*dim] = [hi | lo | hi].
    Returns (split tensor, s).  Elementwise format conversion, not scoring arithmetic."""
    import math
    x = x.float()
    if scale_log2 is None:
        amax = float(x.abs().max().item()) if x.numel() else 0.0
        scale_log2 = int(math.floor(math.log2(32000.0 / amax))) if (amax > 0.0 and math.isfinite(amax)) else 0
    xs = torch.ldexp(x, torch.tensor(scale_log2, device=x.device))
    hi = xs.to(torch.float16)
    lo = (xs - hi.float()).to(torch.float16)
    parts = [hi, lo] if role == "passages" else [hi, lo, hi]
    return torch.cat(parts, dim=1).contiguous(), scale_log2


def flat_ip_topk(queries: torch.Tensor, passages: torch.Tensor, k: int, ids: Optional[torch.Tensor] = None,
                 id_base: int = 0, split_scale: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Exact inner-product top-k of every query against a resident passage shard (faiss IndexFlatIP
    semantics, faiss_indices.py:34).  queries [nq,dim], passages [n,dim] fp16/bf16; returns
    (scores [nq,k] f32 descending, ids [nq,k] int64); ties by id ascending.  1 <= k <= 1024.

    fp32 storage (``token_dtype: float32``): pass ``passages`` = flat_ip_split_f32(p, "passages")[0] ([n, 2*dim] fp16)
    together with its scale as ``split_scale``; queries (fp32 [nq, dim]) are split here, scores are returned unscaled."""
    dev = _require_cuda(queries, passages, ids)
    if passages.dtype not in (torch.float16, torch.bfloat16):
        raise _lib.MatchmakerB200Error("flat_ip_topk: passage storage must be fp16 / bf16, or the fp16 split of fp32 "
                                       "(flat_ip_split_f32)")
    n = passages.shape[0]
    unscale = None
    if split_scale is not None:
        if passages.dtype != torch.float16 or passages.shape[1] % 2:
            raise _lib.MatchmakerB200Error("flat_ip_topk: split storage is [n, 2*dim] fp16")
        dim = passages.shape[1] // 2
        if queries.shape[1] != dim:
            raise _lib.MatchmakerB200Error(f"flat_ip_topk: queries have dim {queries.shape[1]}, split passages {dim}")
        queries, sq = flat_ip_split_f32(queries, "queries")
        unscale = -(sq + split_scale)
        dcode = _lib.F32_SPLIT16
    else:
        queries = queries.to(passages.dtype).contiguous()
        dim = queries.shape[1]
        dcode = _DTYPES[passages.dtype]
    passages = passages.contiguous()
    nq = queries.shape[0]
    if ids is not None:
        ids = ids.to(torch.int64).contiguous()
    lib = _lib.load()
    with torch.cuda.device(dev):
        wsb = lib.mmb200_flat_ip_workspace_bytes(nq, n, k)
        if wsb <= 0:
            raise _lib.MatchmakerB200Error(f"flat_ip_topk: unsupported sizes nq={nq} n={n} k={k} (1 <= k <= {FLAT_IP_MAX_K}): "
                                           + _lib.last_error())
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        out_s = torch.empty((nq, k), dtype=torch.float32, device=dev)
        out_i = torch.empty((nq, k), dtype=torch.int64, device=dev)
        rc = lib.mmb200_flat_ip_topk(_ptr(queries), _ptr(passages), _ptr(ids), _ptr(out_s), _ptr(out_i), _ptr(ws), wsb,
                                     nq, n, dim, k, dcode, id_base, _stream(dev))
    _lib.check(rc, "mmb200_flat_ip_topk")
    if unscale is not None:
        # back to the unscaled domain: a power of two, exact; faiss's "no result" filler (-FLT_MAX) stays what it is
        out_s = torch.where(out_s > -3.0e38, torch.ldexp(out_s, torch.tensor(unscale, device=dev)), out_s)
    return out_s, out_i


def topk_merge(cand_scores: torch.Tensor, cand_ids: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-query merge of candidate lists [nq, L] -> top-k under (score desc, id asc)."""
    dev = _require_cuda(cand_scores, cand_ids)
    cand_scores = cand_scores.to(torch.float32).contiguous()
    cand_ids = cand_ids.to(torch.int64).contiguous()
    nq, L = cand_scores.shape
    out_s = torch.empty((nq, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((nq, k), dtype=torch.int64, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_topk_merge(_ptr(cand_scores), _ptr(cand_ids), _ptr(out_s), _ptr(out_i), nq, L, k, _stream(dev))
    _lib.check(rc, "mmb200_topk_merge")
    return out_s, out_i


def _tkl_slot_map(packed_indices: torch.Tensor) -> torch.Tensor:
    """Packed index of every chunk slot (-1 = dropped by the packing), one kernel launch (mmb200_tkl_slot_map)."""
    pk = packed_indices.reshape(-1)
    if pk.dtype not in (torch.bool, torch.uint8):
        pk = pk != 0
    pk = pk.contiguous()
    out = torch.empty(pk.numel(), dtype=torch.int32, device=pk.device)
    lib = _lib.load()
    with torch.cuda.device(pk.device):
        rc = lib.mmb200_tkl_slot_map(_ptr(pk), _ptr(out), pk.numel(), _stream(pk.device))
    _lib.check(rc, "mmb200_tkl_slot_map")
    return out


def tkl_bwd(q_ctx, q_mask, doc_chunks, chunk_mask, packed_indices, chunk_pieces, mu, sigma, dense_weight, saturation,
            sat_params, sat_red_weight, chunk_scoring, top_idx, orig_score, grad_score):
    """Gradients of the TKL interaction stage: returns (grad_q_ctx, grad_doc_chunks, grad_dense_weight [K],
    grad_chunk_scoring [15], grad_sat_params, grad_sat_red_weight or None)."""
    dev = _require_cuda(q_ctx, doc_chunks, grad_score)
    q_ctx = q_ctx.float().contiguous()
    doc_chunks = doc_chunks.float().contiguous()
    B, Lq, D = q_ctx.shape
    C = int(chunk_pieces)
    slot = _tkl_slot_map(packed_indices)
    q_mask, chunk_mask, mcode = _common_mask_dtype(_prep_mask(q_mask), _prep_mask(chunk_mask))
    mu, sigma, dense_weight = _f32c(mu).view(-1), _f32c(sigma).view(-1), _f32c(dense_weight).view(-1)
    sat_params = _f32c(sat_params).view(-1)
    red = None if sat_red_weight is None else _f32c(sat_red_weight).view(-1)
    K = mu.numel()
    sat_code = {"embedding": 0, "log": 1}[saturation]
    n_sat = 13 if sat_code == 0 else K
    stride = K + 15 + n_sat + (D if sat_code == 0 else 0)
    gq = torch.empty_like(q_ctx)
    gc = torch.empty_like(doc_chunks)
    gp = torch.empty(stride, dtype=torch.float32, device=dev)
    ws = torch.empty(max(1, B) * stride, dtype=torch.float32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.mmb200_tkl_bwd(_ptr(q_ctx), _ptr(q_mask), _ptr(doc_chunks), _ptr(chunk_mask), _ptr(slot), _ptr(mu),
                                _ptr(sigma), _ptr(dense_weight), _ptr(red), _ptr(sat_params),
                                _ptr(_f32c(chunk_scoring).view(-1)), _ptr(top_idx.contiguous()),
                                _ptr(orig_score.contiguous()), _ptr(_f32c(grad_score)), _ptr(gq), _ptr(gc), _ptr(gp),
                                _ptr(ws), B, doc_chunks.shape[0], Lq, D, C, K, sat_code, mcode, _stream(dev))
    _lib.check(rc, "mmb200_tkl_bwd")
    g_dense, g_cs, g_sat = gp[:K], gp[K:K + 15], gp[K + 15:K + 15 + n_sat]
    g_red = gp[K + 15 + n_sat:] if sat_code == 0 else None
    return gq, gc, g_dense, g_cs, g_sat, g_red
