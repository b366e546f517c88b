"""Generate ``tests/golden/*.npz`` by running the reference's OWN classes.

Run in the build container (``/root/reference`` mounted):

    python -m oracle.make_golden

Each fixture stores the seeded inputs, the parameters and the outputs of the
unmodified reference code (imported through ``oracle/reference_loader.py``), and
the script asserts that ``oracle/interaction_oracle.py`` reproduces them before
writing -- that is what pins the oracle.  The fixtures are small and travel to
the GPU box, where the reference itself does not exist.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

from . import interaction_oracle as O
from . import reference_loader as R

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _np(d):
    out = {}
    for k, v in d.items():
        if isinstance(v, torch.Tensor):
            out[k] = v.detach().cpu().numpy()
        else:
            out[k] = np.asarray(v)
    return out


def _save(name, **arrays):
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    np.savez_compressed(path, **_np(arrays))
    print(f"wrote {path} ({os.path.getsize(path) / 1024:.1f} KiB)")


def _check(a, b, what, rtol=1e-6, atol=1e-7):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    err = (a - b).abs().max().item()
    ref = b.abs().max().item()
    assert torch.allclose(a, b, rtol=rtol, atol=atol), f"{what}: oracle != reference (max abs err {err}, ref {ref})"
    print(f"  oracle == reference for {what}: max abs err {err:.3e} (|ref| max {ref:.3e})")


def golden_knrm():
    torch.manual_seed(100)
    for tag, (B, Lq, Ld, D, K) in {"small": (4, 8, 24, 32, 11), "cfg1": (32, 30, 180, 300, 11)}.items():
        ref = R.load_knrm(K)
        q, d, qm, dm = O.synth_kernel_pool_inputs(B, Lq, Ld, D, seed=1235 + Lq)
        with torch.no_grad():
            score, sec = ref.forward(q, d, qm, dm, output_secondary_output=True)
            score_plain = ref.forward(q, d, qm, dm)
        mu = ref.mu.view(-1)
        sigma = ref.sigma.view(-1)
        w = ref.dense.weight.detach().view(-1)
        o_score, o_sec = O.kernel_pool_knrm(q, d, qm, dm, mu, sigma, w)
        _check(o_score, score, f"knrm[{tag}] score")
        _check(o_score, score_plain, f"knrm[{tag}] score (no secondary)")
        _check(o_sec["per_kernel"], sec["per_kernel"], f"knrm[{tag}] per_kernel")
        _check(o_sec["cosine_matrix_masked"], sec["cosine_matrix_masked"], f"knrm[{tag}] cosine")
        assert mu.tolist() == torch.tensor(O.knrm_kernel_mus(K)).tolist()
        assert sigma.tolist() == torch.tensor(O.knrm_kernel_sigmas(K)).tolist()
        _save(f"knrm_{tag}", q=q, d=d, q_mask=qm, d_mask=dm, mu=mu, sigma=sigma, weight=w,
              score=score, per_kernel=sec["per_kernel"], query_mean_vector=sec["query_mean_vector"],
              cosine_matrix_masked=sec["cosine_matrix_masked"])


def golden_tk():
    torch.manual_seed(101)
    emb, heads, layers, ff, max_len = 40, 4, 2, 32, 64
    for tag, (mu, sigma) in {"k11": ([1.0, 0.9, 0.7, 0.5, 0.3, 0.1, -0.1, -0.3, -0.5, -0.7, -0.9], [0.1] * 11),
                             "k21": O.tk_21_kernels()}.items():
        ref = R.load_tk(emb, mu, sigma, heads, layers, ff, max_len, True, True)
        ref.eval()
        with torch.no_grad():
            ref.kernel_alpha_scaler.copy_(torch.rand_like(ref.kernel_alpha_scaler) + 0.5)
        B, Lq, Ld = 5, 12, 48
        q, d, qm, dm = O.synth_kernel_pool_inputs(B, Lq, Ld, emb, seed=2000 + len(mu))
        with torch.no_grad():
            score, sec = ref.forward(q, d, qm, dm, output_secondary_output=True)
            q_ctx = ref.forward_representation(q, qm, ref.positional_features_q[:, :Lq, :])
            d_ctx = ref.forward_representation(d, dm, ref.positional_features_d[:, :Ld, :])
        w = ref.kernel_bin_weights.weight.detach().view(-1)
        alpha = ref.kernel_alpha_scaler.detach().view(-1)
        o_score, o_sec = O.kernel_pool_tk(q_ctx, d_ctx, qm, dm, ref.mu.view(-1), ref.sigma.view(-1), alpha, w)
        _check(o_score, score, f"tk[{tag}] score", rtol=1e-5, atol=1e-6)
        _check(o_sec["per_kernel"], sec["per_kernel"], f"tk[{tag}] per_kernel", rtol=1e-5, atol=1e-5)
        _check(o_sec["cosine_matrix"], sec["cosine_matrix"], f"tk[{tag}] cosine")
        state = {"sd__" + k: v for k, v in ref.state_dict().items()}
        _save(f"tk_{tag}", q=q, d=d, q_mask=qm, d_mask=dm, q_ctx=q_ctx, d_ctx=d_ctx,
              mu=ref.mu.view(-1), sigma=ref.sigma.view(-1), alpha=alpha, weight=w,
              score=score, per_kernel=sec["per_kernel"], query_mean_vector=sec["query_mean_vector"],
              cosine_matrix=sec["cosine_matrix"],
              cfg=np.array([emb, heads, layers, ff, max_len]), **state)


def golden_tkl():
    torch.manual_seed(102)
    emb, heads, layers, ff = 40, 4, 1, 32
    mu = [1.0, 0.9, 0.7, 0.5, 0.3, 0.1, -0.1, -0.3, -0.5, -0.7, -0.9]
    sigma = [0.1] * 11
    for sat in ("embedding", "log"):
        ref = R.load_tkl(emb, mu, sigma, heads, layers, ff, 2000, True, True, sat)
        ref.eval()
        with torch.no_grad():  # make the learned pieces non-trivial but well-conditioned
            ref.chunk_scoring.copy_(torch.rand_like(ref.chunk_scoring) + 0.5)
            ref.kernel_mult.copy_(torch.rand_like(ref.kernel_mult) + 0.5)
            ref.sat_emb_reduce1.weight.copy_(torch.randn_like(ref.sat_emb_reduce1.weight) * 0.3)
            ref.dense.weight.copy_(torch.randn_like(ref.dense.weight) * 0.1)
        B, Lq, Ld = 4, 10, 330
        g = torch.Generator().manual_seed(77)
        q = torch.randn(B, Lq, emb, generator=g) * 0.4
        d = torch.randn(B, Ld, emb, generator=g) * 0.4
        q_len = torch.tensor([10, 7, 3, 10])
        d_len = torch.tensor([330, 200, 47, 121])
        for b in range(B):  # exact matches
            d[b, 5] = q[b, 1]
            d[b, int(d_len[b]) - 3] = q[b, 0]
        qm = (torch.arange(Lq).unsqueeze(0) < q_len.unsqueeze(1)).float()
        dm = (torch.arange(Ld).unsqueeze(0) < d_len.unsqueeze(1)).float()
        q = q * qm.unsqueeze(-1)
        d = d * dm.unsqueeze(-1)
        with torch.no_grad():
            if sat == "embedding":
                score, sec = ref.forward(q, d, qm, dm, output_secondary_output=True)
            else:
                # the reference's secondary-output branch reads `sat_influencer`, which only the
                # "embedding" branch defines (sigir20_tkl.py:290) -> only the score is available
                score, sec = ref.forward(q, d, qm, dm), None
            # the pre-part of forward (sigir20_tkl.py:136-175), re-run to expose the
            # tensors that enter the interaction stage
            q_ctx, _ = ref.forward_representation(q, qm, ref.positional_features_q[:, :Lq, :])
            cd2, cp2, packed, pieces = O.tkl_chunk_documents(d, dm)
            docs_packed = cd2[packed]
            pad_packed = cp2[packed]
            dp, _ = ref.forward_representation(docs_packed, pad_packed,
                                               ref.positional_features_d[:, :docs_packed.shape[1], :])
            doc_chunks_ctx = dp[:, O.TKL_OVERLAP:-O.TKL_OVERLAP, :].contiguous()
            doc_chunk_mask = pad_packed[:, O.TKL_OVERLAP:-O.TKL_OVERLAP].contiguous()
        if sec is not None:
            assert sec["total_chunks"] == cd2.shape[0] and sec["packed_chunks"] == docs_packed.shape[0]
        params = {
            "mu": ref.mu.detach(), "sigma": ref.sigma.detach(), "dense_weight": ref.dense.weight.detach().view(-1),
            "chunk_scoring": ref.chunk_scoring.detach().view(-1),
            "sat_emb_reduce1_weight": ref.sat_emb_reduce1.weight.detach().view(-1),
            "sat_normer_weight": ref.sat_normer.weight.detach(), "sat_normer_bias": ref.sat_normer.bias.detach(),
            "saturation_linear_weight": ref.saturation_linear.weight.detach().view(-1),
            "saturation_linear_bias": ref.saturation_linear.bias.detach(),
            "saturation_linear2_weight": ref.saturation_linear2.weight.detach().view(-1),
            "saturation_linear2_bias": ref.saturation_linear2.bias.detach(),
            "saturation_linear3_weight": ref.saturation_linear3.weight.detach().view(-1),
            "saturation_linear3_bias": ref.saturation_linear3.bias.detach(),
            "kernel_mult0": ref.kernel_mult.detach()[0].view(-1),
        }
        o_score, o_sec = O.tkl_interaction(q_ctx, qm, doc_chunks_ctx, doc_chunk_mask, packed, pieces, params, sat)
        _check(o_score, score, f"tkl[{sat}] score", rtol=1e-5, atol=1e-5)
        if sec is None:  # intermediates come from the (score-pinned) oracle for this branch
            sec = {k: o_sec[k] for k in ("orig_score", "top_non_overlapping_idx", "top_k_non_overlapping")}
        _check(o_sec["orig_score"], sec["orig_score"], f"tkl[{sat}] orig_score", rtol=1e-5, atol=1e-5)
        assert torch.equal(o_sec["top_non_overlapping_idx"], sec["top_non_overlapping_idx"])
        _check(o_sec["top_k_non_overlapping"], sec["top_k_non_overlapping"], f"tkl[{sat}] top15", rtol=1e-5, atol=1e-5)
        state = {"sd__" + k: v for k, v in ref.state_dict().items()
                 if not k.startswith("positional_features")}
        _save(f"tkl_{sat}", q=q, d=d, q_mask=qm, d_mask=dm, q_ctx=q_ctx, doc_chunks_ctx=doc_chunks_ctx,
              doc_chunk_mask=doc_chunk_mask, packed_indices=packed, chunk_pieces=np.array(pieces),
              score=score, orig_score=sec["orig_score"], top_non_overlapping_idx=sec["top_non_overlapping_idx"],
              top_k_non_overlapping=sec["top_k_non_overlapping"],
              cfg=np.array([emb, heads, layers, ff]),
              **{"p__" + k: v for k, v in params.items()}, **state)


def golden_colbert():
    cls, inst = R.load_colbert()
    # (a) fp32, masked pair scoring + unmasked aggregation + all-pairs, small
    q, d, qm, dm = O.synth_colbert_inputs(6, 1, 8, 20, 32, seed=1237, dtype=torch.float32, full_q=False)
    with torch.no_grad():
        score = inst.forward({"vecs": q.clone(), "attention_mask": qm}, {"vecs": d.clone(), "attention_mask": dm},
                             use_fp16=False)
        agg = cls.forward_aggregation(inst, q.clone(), d.clone())
        allp = cls.forward_inbatch_aggregation(inst, q.clone(), qm, d.clone(), dm)
    _check(O.maxsim_pairs(q.clone(), d.clone(), qm, dm), score, "colbert forward (masked)")
    _check(O.maxsim_pairs(q.clone(), d.clone(), None, None), agg, "colbert forward_aggregation")
    _check(O.maxsim_allpairs(q.clone(), qm, d.clone(), dm), allp, "colbert forward_inbatch_aggregation")
    _save("colbert_small", q=q, d=d, q_mask=qm, d_mask=dm, score=score, agg=agg, allpairs=allp)
    # (b) BASELINE config-3 token shape, fp16 storage upcast to fp32 like
    # dense_retrieval.py:406 (.float()), 2 queries x 3 docs
    q, d, qm, dm = O.synth_colbert_inputs(2, 3, 32, 180, 128, seed=1237, dtype=torch.float16)
    qe = q.float().repeat_interleave(3, dim=0)
    qme = qm.repeat_interleave(3, dim=0)
    with torch.no_grad():
        score = inst.forward({"vecs": qe.clone(), "attention_mask": qme},
                             {"vecs": d.float(), "attention_mask": dm}, use_fp16=False)
    _check(O.maxsim_one_query_many_docs(q.float(), d.float(), qm, dm, 3), score, "colbert cfg3-shape")
    _save("colbert_cfg3", q=q, d=d, q_mask=qm, d_mask=dm, docs_per_query=np.array(3), score=score)


def golden_colbert_768():
    """The shape the reference's shipped ColBERT runs at: colbert_compression_dim 768, max_query_length 30,
    max_doc_length 200 (config/train/models/colbert.yaml, config/train/defaults.yaml), fp16 storage upcast to fp32
    like dense_retrieval.py:406; 2 queries x 2 docs."""
    _, inst = R.load_colbert()
    q, d, qm, dm = O.synth_colbert_inputs(2, 2, 30, 200, 768, seed=1768, dtype=torch.float16)
    qe = q.float().repeat_interleave(2, dim=0)
    qme = qm.repeat_interleave(2, dim=0)
    with torch.no_grad():
        score = inst.forward({"vecs": qe.clone(), "attention_mask": qme},
                             {"vecs": d.float(), "attention_mask": dm}, use_fp16=False)
    _check(O.maxsim_one_query_many_docs(q.float(), d.float(), qm, dm, 2), score, "colbert dim-768 shape")
    _save("colbert_768", q=q, d=d, q_mask=qm, d_mask=dm, docs_per_query=np.array(2), score=score)


def golden_bert_dot():
    cls, inst = R.load_bert_dot()
    inst.eval()
    g = torch.Generator().manual_seed(1238)
    qv = torch.randn(8, 64, generator=g)
    dv = torch.randn(8, 64, generator=g)
    with torch.no_grad():
        score = inst.forward({"vecs": qv}, {"vecs": dv}, use_fp16=False)
    _check(O.dot_pairs(qv, dv), score, "bert_dot forward")
    _save("bert_dot_small", qv=qv, dv=dv, score=score)


def golden_tk_sparse():
    """CIKM20_TK_Sparse (models/published/cikm20_tk_sparse.py): full forward of the reference class; the fixture keeps the
    tensors that enter the interaction stage (contextualised embeddings + the learned document-term gate)."""
    torch.manual_seed(103)
    emb, heads, layers, proj, ff, max_len = 40, 4, 1, 16, 32, 64
    mu = [1.0, 0.9, 0.7, 0.5, 0.3, 0.1, -0.1, -0.3, -0.5, -0.7, -0.9]
    sigma = [0.1] * 11
    ref = R.load_tk_sparse(emb, mu, sigma, heads, layers, proj, ff, max_len, True)
    ref.eval()
    with torch.no_grad():
        ref.kernel_alpha_scaler.copy_(torch.rand_like(ref.kernel_alpha_scaler) + 0.5)
        ref.stop_word_reducer2.bias.fill_(0.3)     # so that relu() closes the gate for a share of the document terms
    B, Lq, Ld = 6, 12, 48
    q, d, qm, dm = O.synth_kernel_pool_inputs(B, Lq, Ld, emb, seed=2100)
    with torch.no_grad():
        score, sec, stop = ref.forward(q, d, qm, dm, output_secondary_output=True)
        score_plain, stop_plain = ref.forward(q, d, qm, dm)
        q_ctx, _ = ref.forward_representation(q, qm, ref.positional_features_q[:, :Lq, :])
        d_ctx, _ = ref.forward_representation(d, dm, ref.positional_features_d[:, :Ld, :])
    assert torch.equal(score, score_plain) and torch.equal(stop, stop_plain)
    gate = stop.squeeze(1)
    assert 0.05 < float((gate[dm.bool()] == 0).float().mean()) < 0.95, "the fixture should contain closed and open gates"
    w = ref.kernel_bin_weights.weight.detach().view(-1)
    alpha = ref.kernel_alpha_scaler.detach().view(-1)
    o_score, o_sec = O.kernel_pool_tk_sparse(q_ctx, d_ctx, qm, dm, gate, ref.mu.view(-1), ref.sigma.view(-1), alpha, w)
    _check(o_score, score, "tk_sparse score", rtol=1e-5, atol=1e-6)
    _check(o_sec["per_kernel"], sec["per_kernel"], "tk_sparse per_kernel", rtol=1e-5, atol=1e-5)
    state = {"sd__" + k: v for k, v in ref.state_dict().items()}
    _save("tk_sparse", q=q, d=d, q_mask=qm, d_mask=dm, q_ctx=q_ctx, d_ctx=d_ctx, doc_gate=gate, mu=ref.mu.view(-1),
          sigma=ref.sigma.view(-1), alpha=alpha, weight=w, score=score, per_kernel=sec["per_kernel"],
          document_stop_words=stop, cfg=np.array([emb, heads, layers, proj, ff, max_len]), **state)


def golden_conv_knrm():
    """Conv_KNRM (models/conv_knrm.py): full forward of the reference class + the n-gram tensors between the
    convolutions and the 3 x 3 cross-match."""
    torch.manual_seed(104)
    emb, n_grams, K, conv_out = 24, 3, 11, 32
    ref = R.load_conv_knrm(emb, n_grams, K, conv_out)
    ref.eval()
    B, Lq, Ld = 5, 9, 40
    q, d, qm, dm = O.synth_kernel_pool_inputs(B, Lq, Ld, emb, seed=2200)
    with torch.no_grad():
        score = ref.forward(q, d, qm, dm)
        qg = [c(q.transpose(1, 2)).transpose(1, 2) for c in ref.convolutions]
        dg = [c(d.transpose(1, 2)).transpose(1, 2) for c in ref.convolutions]
    o_score, o_all = O.conv_knrm_cross_match(qg, dg, qm, dm, ref.mu.view(-1), ref.sigma.view(-1), ref.dense.weight.view(-1))
    _check(o_score, score, "conv_knrm score")
    state = {"sd__" + k: v for k, v in ref.state_dict().items()}
    _save("conv_knrm", q=q, d=d, q_mask=qm, d_mask=dm, mu=ref.mu.view(-1), sigma=ref.sigma.view(-1),
          dense_weight=ref.dense.weight.detach().view(-1), score=score, all_grams=o_all,
          cfg=np.array([emb, n_grams, K, conv_out]),
          **{f"qg{i}": t for i, t in enumerate(qg)}, **{f"dg{i}": t for i, t in enumerate(dg)}, **state)


def golden_regen():
    """A second run of the reference's classes on the inputs of committed fixtures (knrm_small, colbert_small, colbert_768):
    tests/test_oracle_golden.py checks the fixtures against it without needing the reference sources."""
    def load(name):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        return {k: torch.from_numpy(z[k]) for k in z.files}

    g = load("knrm_small")
    ref = R.load_knrm(11)
    with torch.no_grad():
        ref.dense.weight.copy_(g["weight"].view(1, -1))
        knrm = ref.forward(g["q"], g["d"], g["q_mask"], g["d_mask"])
    _, inst = R.load_colbert()
    c = load("colbert_small")
    with torch.no_grad():
        colbert = inst.forward({"vecs": c["q"].clone(), "attention_mask": c["q_mask"]},
                               {"vecs": c["d"].clone(), "attention_mask": c["d_mask"]}, use_fp16=False)
    c = load("colbert_768")
    dpq = int(c["docs_per_query"])
    with torch.no_grad():
        colbert_768 = inst.forward({"vecs": c["q"].float().repeat_interleave(dpq, dim=0),
                                    "attention_mask": c["q_mask"].repeat_interleave(dpq, dim=0)},
                                   {"vecs": c["d"].float(), "attention_mask": c["d_mask"]}, use_fp16=False)
    _save("reference_regen", knrm_small_score=knrm, colbert_small_score=colbert, colbert_768_score=colbert_768)


def main():
    if not R.reference_available():
        print("reference not mounted at", R.REFERENCE_ROOT, "- cannot regenerate golden vectors", file=sys.stderr)
        return 1
    only = set(sys.argv[1:])   # e.g. `python -m oracle.make_golden knrm` regenerates one family
    for name, fn in (("knrm", golden_knrm), ("tk", golden_tk), ("tkl", golden_tkl), ("colbert", golden_colbert), ("colbert_768", golden_colbert_768),
                     ("bert_dot", golden_bert_dot), ("tk_sparse", golden_tk_sparse), ("conv_knrm", golden_conv_knrm),
                     ("regen", golden_regen)):
        if not only or name in only:
            fn()
    return 0


if __name__ == "__main__":
    sys.exit(main())
