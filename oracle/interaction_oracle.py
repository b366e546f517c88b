"""CPU restatement (torch, fp32 unless told otherwise) of the reference's
interaction-scoring arithmetic.  TEST INFRASTRUCTURE -- see ``oracle/__init__``.

Every function cites the reference lines it follows (paths relative to
``/root/reference/``).  The op order mirrors the reference so that fp32
round-off matches as closely as a re-implementation can.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch

# ----------------------------------------------------------------------------
# cosine match matrix
# ----------------------------------------------------------------------------


def tiny_value_of_dtype(dtype: torch.dtype) -> float:
    """allennlp.nn.util.tiny_value_of_dtype (allennlp 2.5.1, third party, NOT in
    /root/reference -> parity unpinned): 1e-13 for fp32/fp64, 1e-4 for fp16."""
    if dtype in (torch.float32, torch.float64):
        return 1e-13
    if dtype == torch.float16:
        return 1e-4
    raise TypeError(f"no tiny value for {dtype}")


def cosine_matrix(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """allennlp CosineMatrixAttention.forward (third party, restated): call sites
    matchmaker/models/knrm.py:60, models/published/ecai20_tk.py:105,
    models/published/sigir20_tkl.py:184.

    a [B,Lq,D], b [B,Ld,D] -> [B,Lq,Ld]
    """
    a_norm = a / (a.norm(p=2, dim=-1, keepdim=True) + tiny_value_of_dtype(a.dtype))
    b_norm = b / (b.norm(p=2, dim=-1, keepdim=True) + tiny_value_of_dtype(b.dtype))
    return torch.bmm(a_norm, b_norm.transpose(-1, -2))


# ----------------------------------------------------------------------------
# kernel pooling (KNRM / TK)
# ----------------------------------------------------------------------------


def knrm_kernel_mus(n_kernels: int) -> List[float]:
    """matchmaker/models/knrm.py:101-115."""
    l_mu = [1.0]
    if n_kernels == 1:
        return l_mu
    bin_size = 2.0 / (n_kernels - 1)
    l_mu.append(1 - bin_size / 2)
    for i in range(1, n_kernels - 1):
        l_mu.append(l_mu[i] - bin_size)
    return l_mu


def knrm_kernel_sigmas(n_kernels: int) -> List[float]:
    """matchmaker/models/knrm.py:117-131 (exact-match sigma 1e-4)."""
    bin_size = 2.0 / (n_kernels - 1)
    l_sigma = [0.0001]
    if n_kernels == 1:
        return l_sigma
    l_sigma += [0.5 * bin_size] * (n_kernels - 1)
    return l_sigma


def kernel_pool_knrm(q: torch.Tensor, d: torch.Tensor, q_mask: torch.Tensor, d_mask: torch.Tensor,
                     mu: torch.Tensor, sigma: torch.Tensor, weight: torch.Tensor
                     ) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """KNRM.forward, matchmaker/models/knrm.py:52-84.

    q [B,Lq,D], d [B,Ld,D], masks float {0,1}, mu/sigma [K], weight [K]
    (= ``dense.weight[0]``).  Returns score [B] and the secondary outputs of
    knrm.py:86-88 plus ``per_kernel_query`` (S [B,Lq,K], what backward saves).
    """
    mu = mu.view(1, 1, 1, -1)
    sigma = sigma.view(1, 1, 1, -1)
    qd_mask = torch.bmm(q_mask.unsqueeze(-1), d_mask.unsqueeze(-1).transpose(-1, -2))  # :52
    cos = cosine_matrix(q, d)                                                         # :60
    cos_masked = cos * qd_mask                                                        # :61
    raw = torch.exp(-torch.pow(cos_masked.unsqueeze(-1) - mu, 2) / (2 * torch.pow(sigma, 2)))  # :70
    masked = raw * qd_mask.unsqueeze(-1)                                              # :71
    per_kernel_query = torch.sum(masked, 2)                                           # :73
    log_pkq = torch.log(torch.clamp(per_kernel_query, min=1e-10)) * 0.01              # :74
    log_pkq = log_pkq * q_mask.unsqueeze(-1)                                          # :75
    per_kernel = torch.sum(log_pkq, 1)                                                # :77
    score = per_kernel @ weight.view(-1)                                              # :83-84
    q_mean = q.sum(dim=1) / q_mask.sum(dim=1).unsqueeze(-1)                           # :87
    return score, {"score": score, "per_kernel": per_kernel, "query_mean_vector": q_mean,
                   "cosine_matrix_masked": cos_masked, "per_kernel_query": per_kernel_query}


def kernel_pool_tk(q: torch.Tensor, d: torch.Tensor, q_mask: torch.Tensor, d_mask: torch.Tensor,
                   mu: torch.Tensor, sigma: torch.Tensor, alpha: torch.Tensor, weight: torch.Tensor
                   ) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """ECAI20_TK.forward interaction part, models/published/ecai20_tk.py:105-124.

    q, d are the *contextualised* embeddings (output of forward_representation).
    alpha = ``kernel_alpha_scaler`` [K]; weight = ``kernel_bin_weights.weight[0]``.
    """
    mu = mu.view(1, 1, 1, -1)
    sigma = sigma.view(1, 1, 1, -1)
    cos = cosine_matrix(q, d)                                                          # :105
    raw = torch.exp(-torch.pow(cos.unsqueeze(-1) - mu, 2) / (2 * torch.pow(sigma, 2)))  # :112
    masked = raw * d_mask.unsqueeze(1).unsqueeze(-1)                                   # :114
    per_kernel_query = torch.sum(masked, 2)                                            # :120
    log_pkq = torch.log(torch.clamp(per_kernel_query * alpha.view(1, 1, -1), min=1e-10))  # :121
    log_pkq = log_pkq * q_mask.unsqueeze(-1)                                           # :122
    per_kernel = torch.sum(log_pkq, 1)                                                 # :123
    score = per_kernel @ weight.view(-1)                                               # :124
    q_mean = q.sum(dim=1) / q_mask.sum(dim=1).unsqueeze(-1)                            # :127
    return score, {"score": score, "per_kernel": per_kernel, "query_mean_vector": q_mean,
                   "cosine_matrix": cos * d_mask.unsqueeze(1) * q_mask.unsqueeze(-1),  # :129
                   "per_kernel_query": per_kernel_query}


def kernel_pool_tk_sparse(q: torch.Tensor, d: torch.Tensor, q_mask: torch.Tensor, d_mask: torch.Tensor,
                          doc_stop_words: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, alpha: torch.Tensor,
                          weight: torch.Tensor) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """CIKM20_TK_Sparse.forward interaction part, models/published/cikm20_tk_sparse.py:106-145.

    q, d contextualised embeddings; ``doc_stop_words`` [B, Ld] is the learned per-document-term gate the reference
    computes at :132-133 (``relu(stop_word_reducer2(tanh(stop_word_reducer(.)))) * document_mask``) -- an input here,
    it multiplies every kernel activation of its document term (:135)."""
    mu = mu.view(1, 1, 1, -1)
    sigma = sigma.view(1, 1, 1, -1)
    qd_mask = torch.bmm(q_mask.unsqueeze(-1), d_mask.unsqueeze(-1).transpose(-1, -2))      # :106
    cos = cosine_matrix(q, d)                                                             # :114
    cos_masked = cos * qd_mask                                                            # :115
    raw = torch.exp(-torch.pow(cos_masked.unsqueeze(-1) - mu, 2) / (2 * torch.pow(sigma, 2)))  # :123
    masked = raw * qd_mask.unsqueeze(-1) * doc_stop_words.unsqueeze(1).unsqueeze(-1)       # :135
    per_kernel_query = torch.sum(masked, 2)                                               # :141
    log_pkq = torch.log(torch.clamp(per_kernel_query * alpha.view(1, 1, -1), min=1e-10))  # :142
    log_pkq = log_pkq * q_mask.unsqueeze(-1)                                              # :143
    per_kernel = torch.sum(log_pkq, 1)                                                    # :144
    score = per_kernel @ weight.view(-1)                                                  # :145
    return score, {"score": score, "per_kernel": per_kernel, "cosine_matrix_masked": cos_masked,
                   "per_kernel_query": per_kernel_query}


def conv_knrm_cross_match(q_grams: List[torch.Tensor], d_grams: List[torch.Tensor], q_mask: torch.Tensor,
                          d_mask: torch.Tensor, mu: torch.Tensor, sigma: torch.Tensor, dense_weight: torch.Tensor
                          ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Conv_KNRM.forward after the n-gram convolutions, models/conv_knrm.py:121-170: every query n-gram tensor is
    kernel-pooled against every document n-gram tensor (:125-127 -> forward_matrix_kernel_pooling :144-170, KNRM-style
    masking and the 0.01 log scale), the n*n per-kernel vectors are concatenated (:133) and go through
    ``dense`` = Linear(K*n*n, 1, bias=False) (:135).  Returns (score [B], all_grams [B, n*n*K])."""
    mu4 = mu.view(1, 1, 1, -1)
    sg4 = sigma.view(1, 1, 1, -1)
    qd_mask = torch.bmm(q_mask.unsqueeze(-1), d_mask.unsqueeze(-1).transpose(-1, -2))      # :100
    out = []
    for qg in q_grams:                                                                    # :125
        for dg in d_grams:                                                                # :126
            cos = cosine_matrix(qg, dg) * qd_mask                                         # :151-152
            raw = torch.exp(-torch.pow(cos.unsqueeze(-1) - mu4, 2) / (2 * torch.pow(sg4, 2)))  # :161
            masked = raw * qd_mask.unsqueeze(-1)                                          # :162
            pkq = torch.sum(masked, 2)                                                    # :164
            lpkq = torch.log(torch.clamp(pkq, min=1e-10)) * 0.01                          # :165
            lpkq = lpkq * q_mask.unsqueeze(-1)                                            # :166
            out.append(torch.sum(lpkq, 1))                                                # :168
    all_grams = torch.cat(out, 1)                                                         # :133
    return all_grams @ dense_weight.view(-1), all_grams                                   # :135-138


def idcm_esm_patch_scores(q_ctx: torch.Tensor, d_ctx: torch.Tensor, q_mask: torch.Tensor, d_mask: torch.Tensor,
                          mu: torch.Tensor, sigma: torch.Tensor, alpha: torch.Tensor, weight: torch.Tensor,
                          bias: torch.Tensor) -> torch.Tensor:
    """IDCM's ESM patch scorer, models/published/sigir21_idcm.py:182-186: q_ctx / d_ctx are ALREADY L2-normalised
    (F.normalize, :164-178) so the match matrix is a plain bmm (:182); kernels masked by the patch mask only (:184);
    clamp floor 1e-4 (not 1e-10) on alpha*S (:185); ``sampling_binweights`` = Linear(11, 1, bias=True) (:100, :186).
    PARITY UNPINNED: the class needs HF BERT weights to construct, the lines are restated."""
    cos = torch.bmm(q_ctx, d_ctx.transpose(-1, -2)).unsqueeze(-1)                         # :182
    act = torch.exp(-torch.pow(cos - mu.view(1, 1, 1, -1), 2) / (2 * torch.pow(sigma.view(1, 1, 1, -1), 2))) \
        * d_mask.unsqueeze(-1).unsqueeze(1)                                               # :184
    res = torch.log(torch.clamp(torch.sum(act, 2) * alpha.view(1, 1, -1), min=1e-4)) * q_mask.unsqueeze(-1)  # :185
    return torch.sum(res, 1) @ weight.view(-1) + bias.view(-1)[0]                         # :186


# ----------------------------------------------------------------------------
# ColBERT max-sim
# ----------------------------------------------------------------------------


def maxsim_pairs(q: torch.Tensor, d: torch.Tensor, q_mask: Optional[torch.Tensor],
                 d_mask: Optional[torch.Tensor]) -> torch.Tensor:
    """ColBERT.forward scoring, matchmaker/models/colbert.py:68-75 (masks given),
    and ColBERT.forward_aggregation, colbert.py:100-112 (masks None).

    q [B,Lq,dim], d [B,Ld,dim], masks [B,L] (bool / int attention_mask).
    """
    s = torch.bmm(q, d.transpose(2, 1))                                    # :68 / :101
    if d_mask is not None:
        s[~(d_mask.bool()).unsqueeze(1).expand(-1, s.shape[1], -1)] = -1000  # :69
    s = s.max(-1).values                                                   # :71 / :104
    if q_mask is not None:
        s[~(q_mask.bool())] = 0                                            # :73
    return s.sum(-1)                                                       # :75 / :108


def maxsim_allpairs(q: torch.Tensor, q_mask: torch.Tensor, d: torch.Tensor,
                    d_mask: torch.Tensor) -> torch.Tensor:
    """ColBERT.forward_inbatch_aggregation, matchmaker/models/colbert.py:154-162.

    q [Nq,Lq,dim], d [Nd,Ld,dim] -> [Nq,Nd].
    """
    s = torch.mm(q.reshape(-1, q.shape[-1]), d.reshape(-1, d.shape[-1]).transpose(-2, -1)) \
        .view(q.shape[0], q.shape[1], d.shape[0], d.shape[1])              # :154-155
    s = s.transpose(1, 2)                                                  # :156
    s[~(d_mask.bool()).unsqueeze(1).unsqueeze(1).expand(-1, s.shape[1], s.shape[2], -1)] = -1000  # :158
    s = s.max(-1).values                                                   # :159
    s[~(q_mask.bool()).unsqueeze(1).expand(-1, s.shape[1], -1)] = 0        # :160
    return s.sum(-1)                                                       # :161


def maxsim_allpairs_own_masks(q: torch.Tensor, q_mask: torch.Tensor, d: torch.Tensor,
                              d_mask: torch.Tensor) -> torch.Tensor:
    """All-pairs max-sim with every document masked by ITS OWN mask.  NOT the reference's behaviour:
    colbert.py:158 expands ``document_mask`` [Nd,Ld] over the first (query) axis of the transposed
    [Nq,Nd,Lq,Ld] score tensor, so the reference masks pair (a,b) with the mask of document a
    (see maxsim_allpairs above, which keeps that quirk).  This is the intended semantics, built from
    the pair scorer colbert.py:68-75."""
    out = torch.empty(q.shape[0], d.shape[0], dtype=q.dtype)
    for a in range(q.shape[0]):
        n = d.shape[0]
        out[a] = maxsim_pairs(q[a:a + 1].expand(n, -1, -1), d, q_mask[a:a + 1].expand(n, -1), d_mask)
    return out


def maxsim_one_query_many_docs(q: torch.Tensor, d: torch.Tensor, q_mask: Optional[torch.Tensor],
                               d_mask: Optional[torch.Tensor], docs_per_query: int) -> torch.Tensor:
    """BASELINE config 3 shape ("1 query x 1000 docs, 64 queries"): the reference
    scores it by expanding each query over its documents and calling the pair
    scorer (colbert.py:68-75).  Done per query to bound memory."""
    out = []
    for i in range(q.shape[0]):
        sl = slice(i * docs_per_query, (i + 1) * docs_per_query)
        qi = q[i:i + 1].expand(docs_per_query, -1, -1)
        qm = None if q_mask is None else q_mask[i:i + 1].expand(docs_per_query, -1)
        dm = None if d_mask is None else d_mask[sl]
        out.append(maxsim_pairs(qi, d[sl], qm, dm))
    return torch.cat(out)


# ----------------------------------------------------------------------------
# BERT_DOT
# ----------------------------------------------------------------------------


def dot_pairs(qv: torch.Tensor, dv: torch.Tensor) -> torch.Tensor:
    """BERT_Dot.forward, matchmaker/models/bert_dot.py:62.  qv, dv [B,dim] -> [B]."""
    return torch.bmm(qv.unsqueeze(dim=1), dv.unsqueeze(dim=2)).squeeze(-1).squeeze(-1)


def inbatch_dot(qv: torch.Tensor, dv: torch.Tensor) -> torch.Tensor:
    """In-batch negatives, matchmaker/train.py:439-440: mm(q, d^T) -> [B,B]."""
    return torch.mm(qv, dv.transpose(-2, -1))


def rank_desc_stable(scores: torch.Tensor, ids: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Common tie-break used by BOTH the oracle and the CUDA path when comparing
    top-k: score descending, then id ascending."""
    order_id = torch.argsort(ids, stable=True)
    s1 = scores[order_id]
    order_s = torch.argsort(s1, descending=True, stable=True)
    sel = order_id[order_s][:k]
    return scores[sel], ids[sel]


def flat_ip_search(queries: torch.Tensor, passages: torch.Tensor, ids: torch.Tensor, top_n: int,
                   chunk: int = 262144) -> Tuple[torch.Tensor, torch.Tensor]:
    """Exact max-inner-product search: semantics of ``faiss.IndexIDMap(IndexFlatIP)``
    ``.search`` (faiss-gpu 1.7.0, third party, absent -> PARITY UNPINNED) as called
    at matchmaker/retrieval/faiss_indices.py:27,34 from dense_retrieval.py:391.

    fp32 accumulate, scores descending, returned ids are the user ids given to
    ``add_with_ids``.  faiss leaves tie order unspecified; we fix (score desc,
    id asc).  queries [Nq,dim] fp32, passages [Np,dim] (any float dtype),
    ids [Np] int64.  Returns (scores [Nq,k] f32, ids [Nq,k] i64); slots beyond
    Np are (-inf... faiss uses -3.4e38, id -1).
    """
    nq = queries.shape[0]
    np_ = passages.shape[0]
    k = min(top_n, np_)
    best_s = torch.full((nq, 0), 0.0)
    best_i = torch.zeros((nq, 0), dtype=torch.int64)
    qf = queries.float()
    for lo in range(0, np_, chunk):
        hi = min(np_, lo + chunk)
        s = qf @ passages[lo:hi].float().T
        cand_s = torch.cat([best_s, s], dim=1)
        cand_i = torch.cat([best_i, ids[lo:hi].unsqueeze(0).expand(nq, -1)], dim=1)
        # (score desc, id asc): sort by id first (stable), then by score (stable)
        oi = torch.argsort(cand_i, dim=1, stable=True)
        cs = torch.gather(cand_s, 1, oi)
        ci = torch.gather(cand_i, 1, oi)
        os_ = torch.argsort(cs, dim=1, descending=True, stable=True)[:, :k]
        best_s = torch.gather(cs, 1, os_)
        best_i = torch.gather(ci, 1, os_)
    if k < top_n:
        pad_s = torch.full((nq, top_n - k), -3.4028234663852886e38)
        pad_i = torch.full((nq, top_n - k), -1, dtype=torch.int64)
        best_s = torch.cat([best_s, pad_s], 1)
        best_i = torch.cat([best_i, pad_i], 1)
    return best_s, best_i


def flat_ip_check_exact(queries: torch.Tensor, passages: torch.Tensor, ids: torch.Tensor, got_scores: torch.Tensor,
                        got_ids: torch.Tensor, k: int, chunk_q: int = 64) -> dict:
    """Checker for exact inner-product top-k results against an fp64 ranking.

    The products of fp16 / bf16 values are exact in fp32; what differs between any two fp32 implementations
    (faiss's cuBLAS tiles, torch's CPU sgemm, our tcgen05 chain) is the ORDER of the dim additions.  The fp64 scores
    s64 are the arbiter: with ``tol[q,p] = 4 * sqrt(dim/16) * 2^-24 * sum_i |q_i p_i|`` (a random-walk bound on the
    accumulation error of dim/16 fp32 accumulator updates, x4 margin; the worst case dim * 2^-24 * sum|q_i p_i| is never
    approached)

      * every returned score must lie within tol of s64 of the returned id;
      * rank j of query q is DECIDED when s64 separates it from both fp64 neighbours by more than 2*tol: there the
        returned id must equal the fp64 id, bit-exact;
      * undecided ranks (fp64 near-ties; exact ties are ordered by id ascending in both) may only hold an id from
        their own near-tie run, which for the last ranks extends past k.

    Raises AssertionError on any violation; returns counts for the test log."""
    q64 = queries.double()
    nq, dim = q64.shape
    n = passages.shape[0]
    kk = min(k, n)
    got_scores, got_ids = got_scores.cpu().double(), got_ids.cpu()
    margin = min(n, kk + 64)
    decided = undecided = 0
    for lo in range(0, nq, chunk_q):
        hi = min(nq, lo + chunk_q)
        p64 = passages.double()
        s = q64[lo:hi] @ p64.T                                        # [c, n] fp64
        mass = q64[lo:hi].abs() @ p64.abs().T
        tol = 4.0 * (dim / 16.0) ** 0.5 * 2.0 ** -24 * mass
        # fp64 ranking under (score desc, id asc)
        oi = torch.argsort(ids, stable=True)
        s1, t1 = s[:, oi], tol[:, oi]
        os_ = torch.argsort(s1, dim=1, descending=True, stable=True)[:, :margin]
        rs = torch.gather(s1, 1, os_)
        rt = torch.gather(t1, 1, os_)
        ri = ids[oi][os_]
        for r in range(hi - lo):
            gi, gs = got_ids[lo + r, :kk], got_scores[lo + r, :kk]
            # scores: look the returned id up in the fp64 ranking (it must be inside the margin)
            pos = {int(v): j for j, v in enumerate(ri[r].tolist())}
            gap = (rs[r, :-1] - rs[r, 1:])
            sep = gap > 2.0 * torch.maximum(rt[r, :-1], rt[r, 1:])    # rank j separated from rank j+1
            for j in range(kk):
                g = int(gi[j])
                assert g in pos, f"query {lo + r} rank {j}: id {g} is not among the fp64 top-{margin}"
                jj = pos[g]
                assert abs(gs[j].item() - rs[r, jj].item()) <= rt[r, jj].item(), \
                    f"query {lo + r} rank {j}: score {gs[j].item()} vs fp64 {rs[r, jj].item()} (tol {rt[r, jj].item():.2e})"
                left_ok = j == 0 or bool(sep[j - 1])
                right_ok = j + 1 >= margin or bool(sep[j])
                if left_ok and right_ok:
                    decided += 1
                    assert g == int(ri[r, j]), (f"query {lo + r} rank {j}: id {g} but the fp64 ranking separates id "
                                                f"{int(ri[r, j])} by more than the accumulation bound")
                else:
                    undecided += 1
                    a = j
                    while a > 0 and not bool(sep[a - 1]):
                        a -= 1
                    b = j
                    while b + 1 < margin and not bool(sep[b]):
                        b += 1
                    assert a <= jj <= b, f"query {lo + r} rank {j}: id {g} (fp64 rank {jj}) outside its near-tie run [{a},{b}]"
    if n < k:
        assert (got_ids[:, n:] == -1).all()
    return {"decided": decided, "undecided": undecided}


# ----------------------------------------------------------------------------
# TKL: chunked kernel activations + sliding-window pooling + top-3 hills
# ----------------------------------------------------------------------------

TKL_CHUNK = 40          # sigir20_tkl.py:52
TKL_OVERLAP = 5         # :53
TKL_EXT = TKL_CHUNK + 2 * TKL_OVERLAP  # :54
TKL_WINDOW = 30         # :56
TKL_TOPK = 3            # :57


def tkl_chunk_documents(document_embeddings: torch.Tensor, document_mask: torch.Tensor):
    """sigir20_tkl.py:142-162: pad (5 left, >=10 right), unfold into extended
    chunks of 50 with stride 40, pack the chunks whose 40 centre positions
    contain at least one real token.

    Returns (chunked_docs2 [B*C,50,D], chunked_pad2 [B*C,50], packed_indices
    [B*C] bool, chunk_pieces C).
    """
    ld = document_mask.shape[1]
    if ld > TKL_OVERLAP:
        needed = TKL_EXT - ((ld - TKL_OVERLAP) % TKL_CHUNK)                 # :143
    else:
        needed = TKL_EXT - TKL_OVERLAP - ld                                 # :145
    de = torch.nn.functional.pad(document_embeddings, (0, 0, TKL_OVERLAP, needed))  # :147
    dm = torch.nn.functional.pad(document_mask, (TKL_OVERLAP, needed))      # :148
    chunked_docs = de.unfold(1, TKL_EXT, TKL_CHUNK).transpose(-1, -2)       # :150
    chunked_pad = dm.unfold(1, TKL_EXT, TKL_CHUNK)                          # :151
    chunk_pieces = chunked_docs.shape[1]
    chunked_docs2 = chunked_docs.reshape(-1, TKL_EXT, de.shape[-1])         # :156
    chunked_pad2 = chunked_pad.reshape(-1, TKL_EXT)                         # :157
    packed_indices = chunked_pad2[:, TKL_OVERLAP:-TKL_OVERLAP].sum(-1) != 0  # :159
    return chunked_docs2, chunked_pad2, packed_indices, chunk_pieces


def tkl_interaction(query_ctx: torch.Tensor, query_mask: torch.Tensor,
                    doc_chunks_ctx: torch.Tensor, doc_chunk_mask: torch.Tensor,
                    packed_indices: torch.Tensor, chunk_pieces: int,
                    params: Dict[str, torch.Tensor], saturation: str = "embedding"
                    ) -> Tuple[torch.Tensor, Dict[str, torch.Tensor]]:
    """TKL_sigir20.forward after contextualisation, sigir20_tkl.py:180-286.

    query_ctx [B,Lq,D]      contextualised query embeddings (masked), :136
    doc_chunks_ctx [Nc,40,D] contextualised packed chunks without overlap, :174
    doc_chunk_mask [Nc,40]   :175
    packed_indices [B*C] bool, chunk_pieces C                      :159,:154
    params: mu, sigma [K]; dense_weight [K]; chunk_scoring [15];
            "embedding": sat_emb_reduce1_weight [D], sat_normer_weight/bias [2],
                         saturation_linear{,2,3}_weight [2] / _bias [1]
            "log": kernel_mult0 [K]
    """
    B, Lq, D = query_ctx.shape
    mu = params["mu"].view(1, 1, 1, -1)
    sigma = params["sigma"].view(1, 1, 1, -1)
    K = mu.shape[-1]
    total_chunks = packed_indices.shape[0]
    pq = query_ctx.unsqueeze(1).expand(-1, chunk_pieces, -1, -1).reshape(-1, Lq, D)[packed_indices]  # :180
    cos = cosine_matrix(pq, doc_chunks_ctx)                                               # :184
    raw = torch.exp(-torch.pow(cos.unsqueeze(-1) - mu, 2) / (2 * torch.pow(sigma, 2)))    # :193
    masked = raw * doc_chunk_mask.unsqueeze(1).unsqueeze(-1)                              # :194
    act = torch.zeros((total_chunks, Lq, doc_chunks_ctx.shape[1], K), dtype=query_ctx.dtype)  # :196
    act[packed_indices] = masked                                                          # :197
    act = act.transpose(1, 2).reshape(B, -1, Lq, K).transpose(2, 1)                       # :199  [B,Lq,C*40,K]
    if act.shape[2] < TKL_WINDOW:                                                         # :206
        act = torch.nn.functional.pad(act, (0, 0, 0, TKL_WINDOW - act.shape[2]))
    unrolled = act.unfold(2, TKL_WINDOW, 2).transpose(-1, -2)                             # :209 [B,Lq,W,30,K]
    lengths = torch.sum(unrolled.sum(dim=-1) != 0, dim=-1)                                # :210 [B,Lq,W]
    per_kernel_query = torch.sum(unrolled, -2)                                            # :211 [B,Lq,W,K]

    sat_influencer = None
    if saturation == "embedding":                                                         # :222-234
        red = query_ctx @ params["sat_emb_reduce1_weight"].view(-1, 1)                    # Linear(D,1,no bias)
        sat_influencer = torch.cat([red.expand_as(lengths).unsqueeze(-1),
                                    lengths.float().unsqueeze(-1)], dim=-1)
        sat_influencer = torch.nn.functional.layer_norm(
            sat_influencer, (2,), params["sat_normer_weight"], params["sat_normer_bias"], 1e-5)  # :228
        sat1 = sat_influencer @ params["saturation_linear_weight"].view(2, 1) + params["saturation_linear_bias"]
        sat2 = 1 / (sat_influencer @ params["saturation_linear2_weight"].view(2, 1) + params["saturation_linear2_bias"])
        sat3 = sat_influencer @ params["saturation_linear3_weight"].view(2, 1) + params["saturation_linear3_bias"]
        sat_pkq = sat1 * (torch.clamp(per_kernel_query, min=1e-10) ** sat2) - sat3        # :234
    elif saturation == "log":                                                             # :245-246
        sat_pkq = torch.log(torch.clamp(per_kernel_query * params["kernel_mult0"].view(1, 1, 1, -1), min=1e-10))
    else:
        raise ValueError("reference branches 'idf'/'linear' are dead code (NameError: query_idfs)")

    sat_pkq = sat_pkq * query_mask.unsqueeze(-1).unsqueeze(-1) * (lengths > 0).float().unsqueeze(-1)  # :248
    per_kernel = torch.sum(sat_pkq, 1)                                                    # :249 [B,W,K]
    score = per_kernel @ params["dense_weight"].view(-1)                                  # :251-252 [B,W]
    if score.shape[1] < TKL_TOPK:                                                         # :254
        score = torch.nn.functional.pad(score, (0, TKL_TOPK - score.shape[1]))
    score = score.clone()
    score[score == 0] = -9900                                                             # :257
    orig_score = score
    top_idx, top15 = tkl_top_hills(orig_score)
    orig_score_out = orig_score.clone()
    orig_score_out[orig_score_out <= -9900] = 0                                           # :284
    final = (top15 * params["chunk_scoring"].view(1, -1)).sum(dim=1)                      # :286
    return final, {"score": final, "orig_score": orig_score_out, "top_non_overlapping_idx": top_idx,
                   "top_k_non_overlapping": top15, "per_kernel_query": per_kernel_query,
                   "lengths": lengths, "sat_influencer": sat_influencer}


def tkl_top_hills(orig_score: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """sigir20_tkl.py:263-282: greedy 3x argmax with |r-best| < 15 suppression,
    +-1/+-2 neighbours (clamped), gather 15, sentinel -> 0."""
    B, W = orig_score.shape
    top_idx = torch.zeros((B, TKL_TOPK), dtype=torch.long)
    work = orig_score.clone()
    r = torch.arange(W)
    for c in range(TKL_TOPK):
        best = torch.argmax(work, dim=1)                                                  # :268
        top_idx[:, c] = best
        region = torch.abs(r - best.unsqueeze(-1)) < TKL_WINDOW / 2                       # :270
        work[region] = -10001 - c                                                         # :271
    nb = torch.cat([top_idx, top_idx - 1, top_idx + 1, top_idx - 2, top_idx + 2], dim=1)  # :274
    nb[nb < 0] = 0
    nb[nb >= W] = W - 1
    top15 = torch.gather(orig_score, 1, nb).clone()                                       # :279-280
    top15[top15 <= -9900] = 0                                                             # :281
    return top_idx, top15


# ----------------------------------------------------------------------------
# synthetic MSMARCO-shaped inputs live in matchmaker_b200/synthetic.py (data generation only, shared by
# the tests, bench.py and the golden-vector script); re-exported here for the tests' convenience.
# ----------------------------------------------------------------------------
from matchmaker_b200.synthetic import (synth_colbert_inputs, synth_dense_inputs, synth_kernel_pool_inputs,  # noqa: E402,F401
                                       synth_lengths, tk_21_kernels)
