"""Max-sim across its whole shape envelope against an fp64 restatement of the reference, including the shape the
reference's shipped ColBERT runs at (colbert_compression_dim 768, max_query_length 30, max_doc_length 200, fp16).

Envelope (interaction.maxsim): 1 <= Lq <= 128, 1 <= dim <= 1024, any Ld >= 1, fp16 / bf16 / fp32.  impl="auto" must
return oracle-correct scores everywhere inside it and raise MatchmakerB200Error outside it; a forced impl either matches
the oracle or raises cleanly, never returns wrong numbers.

Tolerance.  fp16 / bf16 products are exact in fp32, so a kernel differs from the fp64 restatement only by fp32 rounding
of the dot products (at most dim * 2^-24 of sum_k |q_k d_k| each) and of the sum over query tokens.  A pair score sums
per-token maxima of either sign, so the repository's 1e-3 bar is applied relative to the magnitude actually summed,
max(|score|, sum_i |max_j s_ij|) -- the same rule as assert_score_close in test_kernel_pool_gpu.py.  A kernel that
picks a wrong row, lets the -1000 fill or a zero-filled padding row win, or drops a token misses it by orders of
magnitude.  The bar is the same for every case.
"""
import pytest
import torch

from conftest import assert_close_rel, load_golden
from matchmaker_b200 import _lib, autograd, interaction
from oracle import interaction_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
REL = 1e-3
ALL_IMPLS = ("auto", "tcgen05", "tcgen05_docm", "tcgen05_ragged", "simt")
FP = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}


def _cuda(*ts):
    return [None if t is None else t.to(DEV) for t in ts]


def _query_slices(n_q, n_d, dpq):
    """(query, first doc, end doc) of every query that owns documents; the last query may own fewer than dpq."""
    return [(i, i * dpq, min((i + 1) * dpq, n_d)) for i in range(n_q) if i * dpq < n_d]


def _token_scores64(q, d, qm, dm, dpq):
    """[n_d, Lq, Ld] fp64 scores of every pair with the reference's -1000 fill of masked document rows
    (colbert.py:68-69), and the [n_d, Lq] query mask of each pair."""
    out, qmask = [], []
    for i, lo, hi in _query_slices(q.shape[0], d.shape[0], dpq):
        s = torch.bmm(q[i:i + 1].double().expand(hi - lo, -1, -1), d[lo:hi].double().transpose(1, 2))
        if dm is not None:
            s = s.masked_fill(~dm[lo:hi].bool().unsqueeze(1), -1000.0)
        out.append(s)
        qmask.append((torch.ones(q.shape[1], dtype=torch.bool) if qm is None else qm[i].bool()).expand(hi - lo, -1))
    return torch.cat(out), torch.cat(qmask)


def ref64(q, d, qm, dm, dpq):
    """(scores, magnitude summed): O.maxsim_pairs on fp64 inputs, one query at a time."""
    scores = []
    for i, lo, hi in _query_slices(q.shape[0], d.shape[0], dpq):
        n = hi - lo
        scores.append(O.maxsim_pairs(q[i:i + 1].double().expand(n, -1, -1), d[lo:hi].double(),
                                     None if qm is None else qm[i:i + 1].expand(n, -1),
                                     None if dm is None else dm[lo:hi]))
    s, qmask = _token_scores64(q, d, qm, dm, dpq)
    mag = (s.max(-1).values.abs() * qmask).sum(-1)
    return torch.cat(scores), mag


def assert_scores(got, ref, what):
    """got within the bar of ref = ref64(...)."""
    ref, mag = ref
    a = got.detach().double().cpu()
    assert a.shape == ref.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(ref.shape)}"
    tol = REL * torch.maximum(ref.abs(), mag)
    err = (a - ref).abs()
    bad = ~(err <= tol)   # NaN counts as bad
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{bad.numel()} pairs off; worst abs err {err.max().item():.3e}, "
                           f"first bad pair {int(bad.nonzero()[0])}: got {a[bad][0].item():.6e} ref {ref[bad][0].item():.6e}")


def assert_valid_argmax(am, q, d, qm, dm, dpq, what):
    """Each argmax entry is a maximiser of its row: its fp64 score lies within fp32 round-off of the fp64 row maximum
    (the kernel and the restatement may order near-ties differently).  It is -1 exactly where the reference sends no
    gradient: masked query tokens, and rows whose maximum is the -1000 fill (or that have no real token)."""
    s, qmask = _token_scores64(q, d, qm, dm, dpq)
    n_d, Lq, Ld = s.shape
    dmask = torch.ones(n_d, Ld, dtype=torch.bool) if dm is None else dm.bool()
    real = s.masked_fill(~dmask.unsqueeze(1), float("-inf"))
    real_max = real.max(-1).values
    fill_wins = dmask.logical_not().any(-1, keepdim=True) & (real_max < -1000.0)
    expect_none = ~qmask | fill_wins | torch.isinf(real_max)
    am = am.cpu().long()
    assert am.shape == (n_d, Lq), f"{what}: argmax shape {tuple(am.shape)}"
    assert (am[expect_none] == -1).all(), f"{what}: argmax set where the reference has no gradient"
    pick = am[~expect_none]
    assert ((pick >= 0) & (pick < Ld)).all(), f"{what}: argmax -1 / out of range where a real row wins"
    # |q| |d|^T: the fp32 round-off bound of each dot product is dim * 2^-24 times this (factor 2 for the tensor pipe's
    # accumulation), summed over the two rows compared
    absdot = torch.cat([torch.bmm(q[i:i + 1].double().abs().expand(hi - lo, -1, -1), d[lo:hi].double().abs().transpose(1, 2))
                        for i, lo, hi in _query_slices(q.shape[0], n_d, dpq)])
    am_c = am.clamp(min=0).unsqueeze(-1)
    best = real.argmax(-1, keepdim=True)
    slack = 2 * q.shape[-1] * 2.0 ** -24 * (absdot.gather(-1, am_c) + absdot.gather(-1, best)).squeeze(-1)
    picked = real.gather(-1, am_c).squeeze(-1)
    ok = picked >= real_max - slack
    assert ok[~expect_none].all(), f"{what}: argmax is not a maximiser ({int((~ok & ~expect_none).sum())} tokens)"


def assert_raises_cleanly(fn, what):
    """A rejected shape raises MatchmakerB200Error with a reason, leaves no CUDA error behind."""
    with pytest.raises(_lib.MatchmakerB200Error) as ei:
        fn()
    msg = str(ei.value)
    assert "CUDA error" not in msg and len(msg.split(":")[-1].strip()) > 0, f"{what}: {msg}"
    torch.cuda.synchronize()


def run_or_reject(fn):
    """Result of fn(), or None if it raised MatchmakerB200Error cleanly (a CUDA error is a failure)."""
    try:
        return fn()
    except _lib.MatchmakerB200Error as e:
        assert "CUDA error" not in str(e), str(e)
        torch.cuda.synchronize()
        return None


def colbert_inputs(n_q, dpq, Lq, Ld, dim, dtype, seed, n_d=None, holes=0.1):
    """Unit-norm token vectors; query lengths in [1, Lq]; document prefix lengths in [1, Ld] with zero, fully padded
    tails; with `holes` > 0 also masked rows inside the prefix; the second document (if any) fully masked."""
    g = torch.Generator().manual_seed(seed)
    n_d = n_q * dpq if n_d is None else n_d
    q = torch.nn.functional.normalize(torch.randn(n_q, Lq, dim, generator=g, dtype=torch.float64), dim=-1)
    d = torch.nn.functional.normalize(torch.randn(n_d, Ld, dim, generator=g, dtype=torch.float64), dim=-1)
    q_len = torch.randint(1, Lq + 1, (n_q,), generator=g)
    d_len = torch.randint(1, Ld + 1, (n_d,), generator=g)
    qm = torch.arange(Lq).unsqueeze(0) < q_len.unsqueeze(1)
    dm = torch.arange(Ld).unsqueeze(0) < d_len.unsqueeze(1)
    if holes > 0:
        dm &= torch.rand(n_d, Ld, generator=g) >= holes
        dm[:, 0] = True
    if n_d > 1:
        dm[1] = False
    q = (q * qm.unsqueeze(-1)).to(dtype)
    d = (d * (torch.arange(Ld).unsqueeze(0) < d_len.unsqueeze(1)).unsqueeze(-1)).to(dtype)
    return q, d, qm, dm


# ---------------------------------------------------------------------------------------------------------------------
# (a) the reference's shipped ColBERT shape: Lq 30, Ld 200, dim 768
# ---------------------------------------------------------------------------------------------------------------------
SHIPPED = dict(Lq=30, Ld=200, dim=768)


@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_shipped_shape_every_impl(dt):
    n_q, dpq = 8, 64
    q, d, qm, dm = colbert_inputs(n_q, dpq, SHIPPED["Lq"], SHIPPED["Ld"], SHIPPED["dim"], FP[dt], seed=768)
    cq, cd, cqm, cdm = _cuda(q, d, qm, dm)
    ref, ref_nomask = ref64(q, d, qm, dm, dpq), ref64(q, d, None, None, dpq)
    for impl in ("auto", "tcgen05", "tcgen05_docm", "simt"):
        got = interaction.maxsim(cq, cd, cqm, cdm, docs_per_query=dpq, impl=impl)
        assert_scores(got, ref, f"{dt} {impl}")
        # unmasked aggregation (colbert.py:100-112)
        got = interaction.maxsim(cq, cd, docs_per_query=dpq, impl=impl)
        assert_scores(got, ref_nomask, f"{dt} {impl} no masks")
    # the ragged fetch lives in the queries-on-M kernel (dim 64 / 128 only)
    assert_raises_cleanly(lambda: interaction.maxsim(cq, cd, cqm, cdm, docs_per_query=dpq, impl="tcgen05_ragged"),
                          "ragged at dim 768")


@pytest.mark.parametrize("impl", ["auto", "tcgen05", "tcgen05_docm", "simt"])
def test_golden_colbert_768(impl):
    """Scores of the reference's own ColBERT class at the shipped shape (oracle/make_golden.py colbert_768)."""
    g = load_golden("colbert_768")
    q, d, qm, dm = _cuda(g["q"], g["d"], g["q_mask"], g["d_mask"])
    dpq = int(g["docs_per_query"])
    s = interaction.maxsim(q, d, qm, dm, docs_per_query=dpq, impl=impl)
    assert_close_rel(s, g["score"], what=f"colbert_768 {impl}")
    assert_scores(s, ref64(g["q"], g["d"], g["q_mask"], g["d_mask"], dpq), f"colbert_768 {impl} vs fp64")


@pytest.mark.parametrize("impl", ["auto", "tcgen05", "tcgen05_docm", "simt"])
def test_allpairs_at_dim_768(impl):
    """In-batch negatives (colbert.py:154-162) with both mask-indexing modes."""
    q, d, qm, dm = colbert_inputs(8, 1, 30, 200, 768, torch.float16, seed=769)
    cq, cd, cqm, cdm = _cuda(q, d, qm, dm)
    qd, dd = q.double(), d.double()
    ref_own = O.maxsim_allpairs_own_masks(qd, qm, dd, dm)
    ref_quirk = O.maxsim_allpairs(qd, qm, dd, dm)
    own = interaction.maxsim_allpairs(cq, cqm, cd, cdm, impl=impl).cpu()
    quirk = interaction.maxsim_allpairs(cq, cqm, cd, cdm, impl=impl, reference_mask_indexing=True).cpu()
    # restate each all-pairs row as pairs so that the summed-magnitude bar applies
    for a in range(8):
        qa = q[a:a + 1].expand(8, -1, -1)
        qma = qm[a:a + 1].expand(8, -1)
        assert_scores(own[a], ref64(qa, d, qma, dm, 8), f"allpairs own masks {impl} row {a}")
        assert_scores(quirk[a], ref64(qa, d, qma, dm[a:a + 1].expand(8, -1), 8), f"allpairs reference indexing {impl} row {a}")
    assert_close_rel(own, ref_own, what="own masks vs O.maxsim_allpairs_own_masks")
    assert_close_rel(quirk, ref_quirk, what="reference indexing vs O.maxsim_allpairs")


def test_host_pipeline_bit_identical_at_dim_768():
    q, d, qm, dm = colbert_inputs(3, 40, 30, 200, 768, torch.float16, seed=770)
    dev = interaction.maxsim(*_cuda(q, d, qm, dm), docs_per_query=40).cpu()
    assert_scores(dev, ref64(q, d, qm, dm, 40), "device path")
    pinned = [t.pin_memory() for t in (q, d, qm, dm)]
    assert torch.equal(interaction.maxsim_host(*pinned, docs_per_query=40), dev)
    assert torch.equal(interaction.maxsim_host(*pinned, docs_per_query=40, chunk_pairs=-1), dev)
    assert torch.equal(interaction.maxsim_host(*pinned, docs_per_query=40, chunk_pairs=7), dev)
    assert torch.equal(interaction.maxsim_host(q, d, qm, dm, docs_per_query=40), dev)


def test_token_index_rerank_at_dim_768():
    import numpy as np
    from matchmaker_b200.retrieval import ColBERTTokenIndex
    g = torch.Generator().manual_seed(771)
    n, dim, Lmax, Lq = 120, 768, 200, 30
    lens = torch.randint(5, Lmax + 1, (n,), generator=g)
    mats = [torch.nn.functional.normalize(torch.randn(int(l), dim, generator=g), dim=-1).half().numpy() for l in lens]
    ext_ids = np.arange(n, dtype=np.int64) * 5 + 1
    idx = ColBERTTokenIndex(dim, Lmax)
    idx.index(ext_ids, mats)
    q = torch.nn.functional.normalize(torch.randn(3, Lq, dim, generator=g), dim=-1).half()
    qm = torch.ones(3, Lq, dtype=torch.bool)
    qm[1, 20:] = False
    cand = torch.stack([torch.randperm(n, generator=g)[:40] for _ in range(3)])
    cand[2, 30:] = -1
    s, ids = idx.rerank(q, qm, cand, top_n=10)
    for qi in range(3):
        ref = []
        for c in cand[qi].tolist():
            if c < 0:
                continue
            dmat = torch.from_numpy(mats[c]).double().unsqueeze(0)
            ref.append((O.maxsim_pairs(q[qi:qi + 1].double(), dmat, qm[qi:qi + 1], None).item(), int(ext_ids[c])))
        ref.sort(key=lambda t: (-t[0], t[1]))
        assert ids[qi].cpu().tolist() == [r[1] for r in ref[:10]]
        assert_close_rel(s[qi].cpu(), torch.tensor([r[0] for r in ref[:10]], dtype=torch.float64), what="rerank scores")


# ---------------------------------------------------------------------------------------------------------------------
# (b) envelope sweep: a pairwise cover of dim x Lq x Ld x dtype
# ---------------------------------------------------------------------------------------------------------------------
SWEEP_DIMS = [64, 96, 100, 128, 192, 320, 384, 448, 512, 576, 768, 1024]
SWEEP_LQ = [1, 31, 32, 33, 64, 65, 96, 97, 128]
SWEEP_LD = [1, 127, 128, 129, 200, 255, 256, 257]
SWEEP_DT = ["fp16", "bf16", "fp32"]
# row (a, b) takes dims[a], Lq[b], Ld[(a + b) % 8], dtype[(a + 2b) % 3]: every pair of values of any two of the four
# parameters occurs in some row (checked below), in 108 cases instead of the 2592 of the full product
SWEEP = [(SWEEP_DIMS[a], SWEEP_LQ[b], SWEEP_LD[(a + b) % 8], SWEEP_DT[(a + 2 * b) % 3])
         for a in range(len(SWEEP_DIMS)) for b in range(len(SWEEP_LQ))]
for _x, _y in [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]:
    _sizes = [len(SWEEP_DIMS), len(SWEEP_LQ), len(SWEEP_LD), len(SWEEP_DT)]
    assert len({(c[_x], c[_y]) for c in SWEEP}) == _sizes[_x] * _sizes[_y], "sweep is not a pairwise cover"


@pytest.mark.parametrize("case", range(len(SWEEP)), ids=[f"dim{c[0]}-Lq{c[1]}-Ld{c[2]}-{c[3]}" for c in SWEEP])
def test_envelope_sweep(case):
    dim, Lq, Ld, dt = SWEEP[case]
    n_q, dpq = 2 + case % 2, 2 + case % 4
    q, d, qm, dm = colbert_inputs(n_q, dpq, Lq, Ld, dim, FP[dt], seed=1000 + case, holes=0.1 if case % 3 else 0.0)
    cq, cd, cqm, cdm = _cuda(q, d, qm, dm)
    what = f"dim {dim} Lq {Lq} Ld {Ld} {dt}"
    ref = ref64(q, d, qm, dm, dpq)
    # inside the envelope auto and simt always serve the shape, with and without argmax
    for impl in ("auto", "simt"):
        assert_scores(interaction.maxsim(cq, cd, cqm, cdm, docs_per_query=dpq, impl=impl), ref, f"{what} {impl}")
    s, am = interaction.maxsim(cq, cd, cqm, cdm, docs_per_query=dpq, return_argmax=True)
    assert_scores(s, ref, f"{what} auto+argmax")
    assert_valid_argmax(am, q, d, qm, dm, dpq, f"{what} auto+argmax")
    # forced tensor-core kernels: correct or a clean refusal
    for impl in ("tcgen05", "tcgen05_docm", "tcgen05_ragged"):
        got = run_or_reject(lambda: interaction.maxsim(cq, cd, cqm, cdm, docs_per_query=dpq, impl=impl))
        if got is not None:
            assert_scores(got, ref, f"{what} {impl}")


def test_outside_envelope_raises():
    for (Lq, dim) in [(129, 64), (129, 768), (30, 1088)]:
        q = torch.zeros(1, Lq, dim, dtype=torch.float16, device=DEV)
        d = torch.zeros(1, 16, dim, dtype=torch.float16, device=DEV)
        for impl in ALL_IMPLS:
            assert_raises_cleanly(lambda: interaction.maxsim(q, d, impl=impl), f"Lq {Lq} dim {dim} {impl}")
        assert_raises_cleanly(lambda: interaction.maxsim(q, d, return_argmax=True), f"Lq {Lq} dim {dim} argmax")


# ---------------------------------------------------------------------------------------------------------------------
# (c) value edges, on each kernel: queries-on-M (dim 128, also with the ragged fetch), the first-generation
# documents-on-M kernel (forced at dim 128; what tcgen05 runs at dim 768), and SIMT at both dims
# ---------------------------------------------------------------------------------------------------------------------
KERNELS = [  # id, dim, impl, produces argmax
    ("qm", 128, "tcgen05", True),
    ("qm_ragged", 128, "tcgen05_ragged", True),
    ("docm", 128, "tcgen05_docm", False),
    ("tc_dim768", 768, "tcgen05", False),
    ("simt128", 128, "simt", True),
    ("simt768", 768, "simt", True),
]
KERNEL_IDS = [k[0] for k in KERNELS]


def _maxsim(k, q, d, qm, dm, dpq, argmax=False):
    _, _, impl, has_argmax = k
    return interaction.maxsim(*_cuda(q, d, qm, dm), docs_per_query=dpq, impl=impl, return_argmax=argmax and has_argmax)


@pytest.mark.parametrize("k", KERNELS, ids=KERNEL_IDS)
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_all_scores_below_fill(k, dt):
    """Every real score below -1000 (vectors of norm ~40 pointing against each other), Ld 300 so that every kernel has
    a part-filled last tile.  No masked row: the true maximum comes back, not the -1000 of the reference's fill and not
    the 0 of a padding row.  One masked row: that -1000 is the maximum of every token, with no gradient."""
    _, dim, _, has_argmax = k
    Lq, Ld, dpq = 30, 300, 3
    g = torch.Generator().manual_seed(dim + Lq)
    e = torch.nn.functional.normalize(torch.randn(dim, generator=g, dtype=torch.float64), dim=0)
    noise = 0.1 / dim ** 0.5   # |noise| ~ 0.1: every score is -1600 * cos(small angle), about -1570
    q = 40 * torch.nn.functional.normalize(e + noise * torch.randn(2, Lq, dim, generator=g, dtype=torch.float64), dim=-1)
    d = -40 * torch.nn.functional.normalize(e + noise * torch.randn(6, Ld, dim, generator=g, dtype=torch.float64), dim=-1)
    q, d = q.to(FP[dt]), d.to(FP[dt])
    qm = torch.ones(2, Lq, dtype=torch.bool)
    qm[1, 25:] = False
    dm = torch.ones(6, Ld, dtype=torch.bool)
    dm[1, 137] = False     # exactly one masked row
    dm[4, 299] = False     # ... in the last tile
    dm[5, 0] = False       # ... first row
    s64, _ = _token_scores64(q, d, None, None, dpq)
    assert (s64 < -1000).all()
    got = _maxsim(k, q, d, qm, None, dpq)
    assert_scores(got, ref64(q, d, qm, None, dpq), f"{k[0]} {dt} no mask")
    got = _maxsim(k, q, d, qm, dm, dpq).cpu()
    assert_scores(got, ref64(q, d, qm, dm, dpq), f"{k[0]} {dt} mask")
    n_tok = qm.repeat_interleave(dpq, 0).sum(-1).float()
    for p in (1, 4, 5):
        assert got[p].item() == -1000.0 * n_tok[p].item(), f"{k[0]}: pair {p} {got[p].item()}"
    for p in (0, 2, 3):
        assert got[p].item() < -1000.0 * n_tok[p].item() - 100
    if has_argmax:
        s, am = _maxsim(k, q, d, qm, dm, dpq, argmax=True)
        assert torch.equal(s.cpu(), got)
        assert_valid_argmax(am, q, d, qm, dm, dpq, k[0])
        assert (am.cpu()[[1, 4, 5]] == -1).all()


@pytest.mark.parametrize("k", KERNELS, ids=KERNEL_IDS)
def test_exact_ties_take_the_first_row(k):
    """Each query token's best row occurs four times (bit-identical rows, in different warps / tiles of every kernel):
    the argmax is the first occurrence; masking it moves the argmax to the second."""
    _, dim, _, has_argmax = k
    Lq, Ld, dpq = 30, 300, 2
    g = torch.Generator().manual_seed(7 * dim)
    q = torch.nn.functional.normalize(torch.randn(1, Lq, dim, generator=g), dim=-1).half()
    d = (0.05 * torch.nn.functional.normalize(torch.randn(2, Ld, dim, generator=g), dim=-1)).half()
    starts = (7, 71, 150, 260)
    for s0 in starts:
        d[:, s0:s0 + Lq] = q[0]
    dm = torch.ones(2, Ld, dtype=torch.bool)
    dm[1, 7:7 + Lq] = False    # first copies masked in document 1: the second copies win
    got = _maxsim(k, q, d, None, dm, dpq)
    assert_scores(got, ref64(q, d, None, dm, dpq), f"{k[0]} ties")
    if has_argmax:
        s, am = _maxsim(k, q, d, None, dm, dpq, argmax=True)
        assert torch.equal(s, got)
        tok = torch.arange(Lq, dtype=torch.int32)
        assert torch.equal(am.cpu(), torch.stack([7 + tok, 71 + tok])), f"{k[0]}: {am.cpu()}"


@pytest.mark.parametrize("k", KERNELS, ids=KERNEL_IDS)
def test_fp16_products_beyond_fp16_range(k):
    """Entries of magnitude 260..300: every product exceeds the fp16 maximum (65504), the fp32 accumulator holds it."""
    _, dim, _, has_argmax = k
    Lq, Ld, dpq = 30, 200, 2
    g = torch.Generator().manual_seed(11 * dim)

    def big(*shape):
        mag = 260 + 40 * torch.rand(*shape, generator=g)
        return torch.where(torch.rand(*shape, generator=g) < 0.5, -mag, mag).half()
    q, d = big(2, Lq, dim), big(4, Ld, dim)
    qm = torch.ones(2, Lq, dtype=torch.bool)
    dm = torch.arange(Ld).unsqueeze(0) < torch.tensor([[200], [150], [9], [1]])
    got = _maxsim(k, q, d, qm, dm, dpq)
    assert torch.isfinite(got).all()
    assert_scores(got, ref64(q, d, qm, dm, dpq), f"{k[0]} fp16 overflow")
    if has_argmax:
        s, am = _maxsim(k, q, d, qm, dm, dpq, argmax=True)
        assert torch.equal(s, got)
        assert_valid_argmax(am, q, d, qm, dm, dpq, f"{k[0]} fp16 overflow")


def _bwd_ref64(q, d, am, grad, dpq):
    """fp64 gradients of the oracle expression at the given argmax: grad_q[qi,i] = sum_p g_p d[p, a_pi],
    grad_d[p, j] = sum_{i: a_pi = j} g_p q[qi, i]; and the magnitudes summed into each entry."""
    n_d, Ld = d.shape[0], d.shape[1]
    gq, gd = torch.zeros(q.shape, dtype=torch.float64), torch.zeros(d.shape, dtype=torch.float64)
    mq, md = torch.zeros_like(gq), torch.zeros_like(gd)
    am = am.cpu().long()
    for i, lo, hi in _query_slices(q.shape[0], n_d, dpq):
        for p in range(lo, hi):
            a = am[p]
            onehot = ((a.unsqueeze(1) == torch.arange(Ld).unsqueeze(0)) & (a >= 0).unsqueeze(1)).double()  # [Lq, Ld]
            gp = float(grad[p])
            gq[i] += gp * onehot @ d[p].double()
            mq[i] += abs(gp) * onehot @ d[p].double().abs()
            gd[p] = gp * onehot.T @ q[i].double()
            md[p] = abs(gp) * onehot.T @ q[i].double().abs()
    return gq, gd, mq, md


def _assert_grad(got, ref, mag, what):
    a = got.detach().double().cpu()
    tol = REL * torch.maximum(ref.abs(), mag)
    err = (a - ref).abs()
    assert (err <= tol).all(), f"{what}: {int((err > tol).sum())}/{err.numel()} off, worst {err.max().item():.3e}"


def _check_backward(q, d, qm, dm, dpq, what):
    """Forward argmax is a valid maximiser; the fp32 backward equals the fp64 gradient at that argmax; autograd returns
    it cast to the input dtype and is bit-identical run to run."""
    cq, cd, cqm, cdm = _cuda(q, d, qm, dm)
    s, am = interaction.maxsim(cq, cd, cqm, cdm, docs_per_query=dpq, return_argmax=True)
    assert_scores(s, ref64(q, d, qm, dm, dpq), f"{what} forward")
    assert_valid_argmax(am, q, d, qm, dm, dpq, what)
    grad = torch.randn(d.shape[0], generator=torch.Generator().manual_seed(5), dtype=torch.float64).float()
    gq, gd = interaction.maxsim_bwd(cq, cd, grad.to(DEV), am, docs_per_query=dpq)
    rq, rd, mq, md = _bwd_ref64(q, d, am, grad, dpq)
    _assert_grad(gq, rq, mq, f"{what} grad_q")
    _assert_grad(gd, rd, md, f"{what} grad_d")
    runs = []
    for _ in range(2):
        xq, xd = cq.clone().requires_grad_(True), cd.clone().requires_grad_(True)
        out = autograd.maxsim(xq, xd, cqm, cdm, docs_per_query=dpq)
        out.backward(grad.to(DEV))
        runs.append((out.detach(), xq.grad, xd.grad))
    assert torch.equal(runs[0][0], s)
    assert torch.equal(runs[0][1], gq.to(q.dtype)) and torch.equal(runs[0][2], gd.to(d.dtype))
    assert all(torch.equal(x, y) for x, y in zip(runs[0], runs[1])), f"{what}: two runs differ"


@pytest.mark.parametrize("dim", [128, 768])
def test_short_last_query(dim):
    """n_d not a multiple of docs_per_query: the last query owns fewer documents, forward on every kernel and backward."""
    n_q, dpq, n_d = 3, 4, 10
    q, d, qm, dm = colbert_inputs(n_q, dpq, 30, 200, dim, torch.float16, seed=dim + 3, n_d=n_d)
    ref = ref64(q, d, qm, dm, dpq)
    for k in KERNELS:
        if k[1] == dim:
            assert_scores(_maxsim(k, q, d, qm, dm, dpq), ref, f"{k[0]} short last query")
    _check_backward(q, d, qm, dm, dpq, f"dim {dim} short last query")


def _misaligned(t):
    """A contiguous view of t whose storage starts one element (2 bytes for fp16 / bf16) past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=DEV)
    v = buf[1:].view(t.shape)
    v.copy_(t.to(DEV))
    assert v.is_contiguous() and v.data_ptr() % 16 == t.element_size()
    return v


@pytest.mark.parametrize("dim", [128, 768])
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_misaligned_storage(dim, dt):
    """q / d not 16-byte aligned: the TMA kernels refuse them, auto falls back and stays correct, forward and backward."""
    dpq = 3
    q, d, qm, dm = colbert_inputs(2, dpq, 30, 200, dim, FP[dt], seed=dim + 4)
    mq, md = _misaligned(q), _misaligned(d)
    cqm, cdm = _cuda(qm, dm)
    ref = ref64(q, d, qm, dm, dpq)
    for impl in ("auto", "simt"):
        assert_scores(interaction.maxsim(mq, md, cqm, cdm, docs_per_query=dpq, impl=impl), ref, f"misaligned {impl}")
    for impl in ("tcgen05", "tcgen05_docm", "tcgen05_ragged"):
        assert_raises_cleanly(lambda: interaction.maxsim(mq, md, cqm, cdm, docs_per_query=dpq, impl=impl),
                              f"misaligned {impl}")
    s, am = interaction.maxsim(mq, md, cqm, cdm, docs_per_query=dpq, return_argmax=True)
    assert_scores(s, ref, "misaligned auto+argmax")
    assert_valid_argmax(am, q, d, qm, dm, dpq, "misaligned argmax")
    grad = torch.randn(d.shape[0], generator=torch.Generator().manual_seed(6)).to(DEV)
    gq, gd = interaction.maxsim_bwd(mq, md, grad, am, docs_per_query=dpq)
    rq, rd, mgq, mgd = _bwd_ref64(q, d, am, grad.cpu(), dpq)
    _assert_grad(gq, rq, mgq, "misaligned grad_q")
    _assert_grad(gd, rd, mgd, "misaligned grad_d")


# ---------------------------------------------------------------------------------------------------------------------
# (d) training at the shipped shape
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dpq", [1, 8])
@pytest.mark.parametrize("dt", ["fp16", "bf16", "fp32"])
def test_training_at_dim_768(dt, dpq):
    n_q = 8 if dpq == 1 else 3
    q, d, qm, dm = colbert_inputs(n_q, dpq, SHIPPED["Lq"], SHIPPED["Ld"], SHIPPED["dim"], FP[dt], seed=772 + dpq)
    _check_backward(q, d, qm, dm, dpq, f"{dt} dpq {dpq}")
