#!/usr/bin/env python
"""Benchmark of the interaction-scoring hot path (BASELINE.json metric: query-doc pairs scored / s,
ColBERT max-sim, dim=128, Lq=32, Ld=180, 64 queries x 1000 docs per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload colbert|tk|knrm|tkl|bert_dot]     (default colbert = the BASELINE metric)
                    [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL).  Prints ONE JSON line on rank 0.

A "step" = one pass of the hot path over one synthetic batch (workload below).  `value` is whole-job
pairs/s with inputs resident in HBM; `e2e` is the same metric through the host-buffer C-ABI call
(pinned host inputs -> H2D -> kernel -> D2H scores inside the timed region); `roofline` is the max-sim
kernel's algorithmic bytes / its CUDA-event duration against the measured HBM peak; `cpu_baseline` is
the CPU oracle (port of the reference's PyTorch path, timed on this host's cores).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# BASELINE config 3
N_QUERIES, DOCS_PER_QUERY, LQ, LD, DIM = 64, 1000, 32, 180, 128
SEED = 1237
TOPK = 100
# SURVEY.md 8(d): doc tile Ld*dim*2 + 4 B length + 4 B score + query tile amortised over 1000 docs
ALG_BYTES_PER_PAIR = LD * DIM * 2 + 4 + 4 + (LQ * DIM * 2) // DOCS_PER_QUERY
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent


def _tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            pass
    return 1400.0, "fallback (B200_PROFILING.md sustained)"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled every ~5 ms through NVML while the timed regions run (nvidia-smi
    -lms 200 is too coarse: the 20-step timed region of this kernel lasts ~10 ms)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            idx = self.gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag.is_set():
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = get_reasons(self.h)
                self.samples.append((time.perf_counter(), clk, rs))
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                break
            time.sleep(0.005)

    def stop(self, windows):
        """windows: list of (t0, t1) perf_counter intervals that were timed regions."""
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        self.stop_flag.set()
        self.thread.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)]
        used = inside if inside else self.samples
        clocks = [c for _, c, _ in used]
        reasons = set()
        for _, _, r in used:
            for n, bit in names.items():
                if r & bit:
                    reasons.add(n)
        return {"sm_mhz": statistics.median(clocks) if clocks else None, "sm_max_mhz": self.smax,
                "samples_in_timed_regions": len(inside), "samples_total": len(self.samples),
                "reasons": sorted(reasons), "how": "NVML poll every 5 ms; timed regions = value loop + e2e loop"}


# ------------------------------------------------------------------------------------------------------------
# workloads (BASELINE.json configs).  Each one: synthetic seeded inputs of that config's shape, a GPU step on
# HBM-resident inputs, an end-to-end step from pinned host buffers, the CPU oracle step, algorithmic bytes.
# ------------------------------------------------------------------------------------------------------------
class ColbertWorkload:
    """BASELINE config 3: ColBERT max-sim, dim=128, Lq=32, Ld=180, 64 queries x 1000 docs per GPU, fp16.

    N > 1 is a sharded search of ONE query set: every rank holds the same 64 queries (seed SEED) and its own
    1000-document shard per query (seed SEED + 1 + rank); the per-query top-100 is exchanged and merged.
    Documents are generated on the GPU (unit-norm randn rows, MSMARCO-shaped lengths, zero padding, fp16) so that a
    rank never holds more than the 2.95 GB fp16 copy in host memory (8 ranks generating 5.9 GB fp32 temporaries each
    on the host cores is what a shared box does not need); the CPU legs read that same tensor back."""
    name = "colbert_maxsim"
    metric = "query-doc pairs scored/sec (ColBERT max-sim d=128)"
    dtype = "f16"
    kernel = "maxsim_qm_kernel"
    bound = "hbm"
    launches_per_step = 1

    def __init__(self, rank, dev):
        from matchmaker_b200 import synthetic as O
        self.dev = dev
        self.rank = rank
        g = torch.Generator().manual_seed(SEED)
        q = torch.nn.functional.normalize(torch.randn(N_QUERIES, LQ, DIM, generator=g), dim=-1)
        self.q = q.to(torch.float16)
        self.qm = torch.ones(N_QUERIES, LQ, dtype=torch.bool)   # MASK-augmented queries are always full length
        gl = torch.Generator().manual_seed(SEED + 1 + rank)
        self.d_len = O.synth_lengths(N_QUERIES * DOCS_PER_QUERY, 75.0, 30.0, 10, LD, gl)
        self.pairs = N_QUERIES * DOCS_PER_QUERY
        self.alg_bytes = ALG_BYTES_PER_PAIR * self.pairs
        self.alg_note = "SURVEY 8(d): Ld*dim*2 + 4 + 4 + Lq*dim*2/docs_per_query = %d B/pair" % ALG_BYTES_PER_PAIR
        self.id_base = rank * self.pairs
        self.d = None

    def _generate_docs(self, dev):
        n = self.pairs
        dm = torch.arange(LD, device=dev).unsqueeze(0) < self.d_len.to(dev).unsqueeze(1)
        d = torch.empty((n, LD, DIM), dtype=torch.float16, device=dev)
        gg = torch.Generator(device=dev).manual_seed(SEED + 1 + self.rank)
        step = 8000
        for lo in range(0, n, step):   # bounded temporaries: 8000 x 180 x 128 fp32 = 737 MB
            x = torch.randn((min(step, n - lo), LD, DIM), generator=gg, device=dev)
            x = torch.nn.functional.normalize(x, dim=-1) * dm[lo:lo + step].unsqueeze(-1)
            d[lo:lo + step] = x.to(torch.float16)
        return d, dm

    def to_device(self):
        dev = self.dev
        self.cq, self.cqm = self.q.to(dev), self.qm.to(dev)
        self.cd, self.cdm = self._generate_docs(dev)

    def kernel_step(self):
        from matchmaker_b200 import interaction
        return interaction.maxsim(self.cq, self.cd, self.cqm, self.cdm, docs_per_query=DOCS_PER_QUERY, impl="tcgen05")

    def outputs(self, out):
        return {"scores": out}

    def exchange(self, s):
        from matchmaker_b200 import sharding
        return sharding.topk_all_gather_merge(s.view(N_QUERIES, DOCS_PER_QUERY), TOPK, self.id_base)

    def _host_copy(self):
        if self.d is not None:
            return
        if not hasattr(self, "cd"):
            # reference arm (no device copy exists): same generator on the GPU when the box has one -- the data are
            # then identical to the GPU arm's -- else on the host cores
            gdev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
            d, dm = self._generate_docs(gdev)
            self.d, self.dm = d.cpu(), dm.cpu()
            return
        self.d = torch.empty(self.cd.shape, dtype=self.cd.dtype, pin_memory=True)
        self.d.copy_(self.cd)
        self.dm = torch.empty(self.cdm.shape, dtype=torch.bool, pin_memory=True)
        self.dm.copy_(self.cdm)
        torch.cuda.synchronize()

    def pin(self):
        """Pinned host buffers of the end-to-end call.  Returns the bytes one e2e step really moves host->device:
        mmb200_maxsim_fwd_host takes the zero-copy path for pinned documents -- the kernel's TMA reads each document
        over PCIe in 16-row blocks up to its last unmasked row -- so padding rows never travel."""
        self._host_copy()
        self.h = [self.q.pin_memory(), self.d, self.qm.pin_memory(), self.dm]
        rows16 = ((self.d_len + 15) // 16) * 16
        fetched = int(rows16.sum().item()) * DIM * 2
        small = self.h[0].numel() * 2 + self.h[2].numel() + self.h[3].numel()
        self.h2d_dense = sum(x.numel() * x.element_size() for x in self.h)
        return fetched + small

    def e2e_step(self):
        from matchmaker_b200 import interaction
        return interaction.maxsim_host(*self.h, docs_per_query=DOCS_PER_QUERY, device=self.dev)

    def e2e_pageable_step(self):
        """Same call on PAGEABLE host tensors: no zero-copy, the library stages 96 MB slabs through its own
        buffers (cudaMemcpyAsync from pageable memory) -- what a caller that never pins would see."""
        from matchmaker_b200 import interaction
        if not hasattr(self, "pg"):
            self.pg = [x.clone() for x in (self.q, self.d, self.qm, self.dm)]   # clone() of a pinned tensor is pageable
        return interaction.maxsim_host(*self.pg, docs_per_query=DOCS_PER_QUERY, device=self.dev)

    e2e_note = ("mmb200_maxsim_fwd_host on pinned host tensors: q + masks copied (cudaMemcpyAsync), documents read by the "
                "kernel's TMA straight from pinned host memory over PCIe (zero-copy, 16-row blocks up to each document's "
                "last unmasked row), scores copied back; h2d_bytes_per_step counts the bytes that really cross PCIe, "
                "h2d_bytes_dense is the size of the host tensors; pinning happens once, outside the timed region")

    def cpu_prepare(self):
        self._host_copy()
        self.cpu_n = N_QUERIES   # one CPU step = the whole workload (64 000 pairs), as in the GPU arm
        nd = self.cpu_n * DOCS_PER_QUERY
        self.q32, self.d32 = self.q[:self.cpu_n].float(), self.d[:nd].float()  # dense_retrieval.py:406 upcasts fp16 storage
        self.cqm_l, self.cdm_l = self.qm[:self.cpu_n].long(), self.dm[:nd].long()

    def cpu_pairs(self):
        return self.cpu_n * DOCS_PER_QUERY

    def cpu_step(self):
        from oracle import interaction_oracle as O
        with torch.no_grad():
            return O.maxsim_one_query_many_docs(self.q32, self.d32, self.cqm_l, self.cdm_l, DOCS_PER_QUERY)

    def config(self, n_gpus):
        return {"workload": self.name, "queries_per_gpu": N_QUERIES, "docs_per_query": DOCS_PER_QUERY, "Lq": LQ,
                "Ld": LD, "dim": DIM, "storage_dtype": "float16", "mask_dtype": "bool",
                "pairs_per_step": self.pairs * n_gpus,
                "sharding": "documents sharded over ranks (same 64 queries on every rank); per-query top-%d "
                            "all-gather + merge when N>1" % TOPK,
                "l2_policy": "inputs larger than L2 (2.95 GB of documents per GPU per step vs 126 MB L2)"}


class KernelPoolWorkload:
    """BASELINE config 2 (TK interaction: Lq=30, Ld=200, D=300, 21 kernels) or config 1 shape (KNRM: Ld=180, 11
    kernels); op-level: the contextualised embeddings are the inputs.  The batch is enlarged (default 4096 pairs
    = 16 x the config's batch of 256) so that the inputs (1.1 GB) exceed L2."""
    bound = "hbm"
    dtype = "f32"
    launches_per_step = 1

    def __init__(self, rank, dev, kind):
        from matchmaker_b200 import synthetic as O
        from matchmaker_b200.rankers.knrm import kernel_mus, kernel_sigmas
        self.dev, self.kind = dev, kind
        if kind == "tk":
            self.name, self.B, self.Lq, self.Ld, self.D = "tk_kernel_pool", 4096, 30, 200, 300
            mu, sg = O.tk_21_kernels()
            self.log_scale, self.alpha = 1.0, torch.linspace(0.5, 1.5, 21)
        else:
            self.name, self.B, self.Lq, self.Ld, self.D = "knrm_kernel_pool", 4096, 30, 180, 300
            mu, sg = kernel_mus(11), kernel_sigmas(11)
            self.log_scale, self.alpha = 0.01, None
        self.metric = "query-doc pairs scored/sec (%s cosine + RBF kernel pooling forward, D=300)" % kind.upper()
        self.kernel = "kernel_pool_ts_kernel"
        self.mu, self.sigma = torch.tensor(mu), torch.tensor(sg)
        self.w = torch.linspace(-0.014, 0.014, len(mu))
        self.q, self.d, self.qm, self.dm = O.synth_kernel_pool_inputs(self.B, self.Lq, self.Ld, self.D, seed=SEED + 10 + rank)
        self.pairs = self.B
        per_pair = (self.Lq + self.Ld) * self.D * 4 + (self.Lq + self.Ld) * 4 + 4
        self.alg_bytes = per_pair * self.B
        self.alg_note = "SURVEY 8(d): (Lq+Ld)*D*4 + (Lq+Ld)*4 + 4 = %d B/pair" % per_pair

    def to_device(self):
        d = self.dev
        self.c = [t.to(d) for t in (self.q, self.d, self.qm, self.dm, self.mu, self.sigma, self.w)]
        self.calpha = None if self.alpha is None else self.alpha.to(d)

    def kernel_step(self):
        from matchmaker_b200 import interaction
        return interaction.kernel_pool(*self.c, alpha=self.calpha, log_scale=self.log_scale)["score"]

    def outputs(self, out):
        return {"scores": out}

    def exchange(self, s):
        return s  # re-ranking pairs are independent: no data-path collective

    def pin(self):
        self.h = [t.pin_memory() for t in (self.q, self.d, self.qm, self.dm)]
        return sum(x.numel() * x.element_size() for x in self.h)

    def e2e_step(self):
        from matchmaker_b200 import interaction
        dq, dd, dqm, ddm = [t.to(self.dev, non_blocking=True) for t in self.h]
        s = interaction.kernel_pool(dq, dd, dqm, ddm, *self.c[4:], alpha=self.calpha, log_scale=self.log_scale)["score"]
        return s.cpu()

    e2e_note = "pinned host embeddings+masks -> H2D -> mmb200_kernel_pool_fwd -> D2H scores (the eval.py:89-161 pattern)"

    def cpu_prepare(self):
        self.cpu_n = 256  # the config's own batch size

    def cpu_step(self):
        from oracle import interaction_oracle as O
        n = self.cpu_n
        with torch.no_grad():
            if self.kind == "tk":
                return O.kernel_pool_tk(self.q[:n], self.d[:n], self.qm[:n], self.dm[:n], self.mu, self.sigma, self.alpha, self.w)[0]
            return O.kernel_pool_knrm(self.q[:n], self.d[:n], self.qm[:n], self.dm[:n], self.mu, self.sigma, self.w)[0]

    def config(self, n_gpus):
        return {"workload": self.name, "pairs_per_gpu": self.B, "Lq": self.Lq, "Ld": self.Ld, "dim": self.D,
                "kernels": int(self.mu.numel()), "pairs_per_step": self.B * n_gpus,
                "sharding": "pairs split over ranks, no collective",
                "l2_policy": "inputs larger than L2 (%.2f GB per GPU per step)" % (self.alg_bytes / 1e9)}


class KernelPoolTrainWorkload(KernelPoolWorkload):
    """TK interaction forward + backward (what train.py:504,526 runs per step through autograd): scores, then gradients
    to both embedding tensors, alpha and the bin weights.  Algorithmic bytes per pair (SURVEY 8(d) K2 row): the forward
    reads q, d, masks; the backward reads them again plus S [Lq, K] and writes dq, dd."""
    launches_per_step = 3   # forward (saves cosines + norms), tcgen05 backward, batch reduction of d weight / d alpha
    graph_ok = True         # torch.autograd inside the capture (forward + backward of the step, as in whole-step capture)

    def __init__(self, rank, dev, pairs=1024):
        super().__init__(rank, dev, "tk")
        self.name = "tk_kernel_pool_train"
        self.B = self.pairs = pairs   # <= the 4096 pairs of the forward workload
        self.q, self.d, self.qm, self.dm = self.q[:self.B], self.d[:self.B], self.qm[:self.B], self.dm[:self.B]
        self.metric = "query-doc pairs/sec (TK cosine + RBF kernel pooling forward + backward, D=300)"
        self.kernel = "kernel_pool_ts_kernel<save> + kernel_pool_bwd_tc_kernel"
        fwd = (self.Lq + self.Ld) * self.D * 4 + (self.Lq + self.Ld) * 4 + 4
        bwd = fwd + self.Lq * 21 * 4 * 2 + (self.Lq + self.Ld) * self.D * 4
        saved = (33 * self.Ld + 32) * 4 * 2   # cosines + inverse norms: written by the forward, read by the backward
        self.alg_bytes = (fwd + bwd + saved) * self.B
        self.alg_note = ("forward %d B/pair + backward %d B/pair (inputs re-read, S saved and re-read, dq/dd written) + %d B/pair of "
                         "saved cosines / norms (written + read)" % (fwd, bwd, saved))

    def to_device(self):
        super().to_device()
        self.c[0].requires_grad_(True)
        self.c[1].requires_grad_(True)
        self.c[6].requires_grad_(True)
        self.calpha.requires_grad_(True)
        self.gout = torch.ones(self.B, device=self.dev)

    def kernel_step(self):
        from matchmaker_b200 import autograd
        for t in (self.c[0], self.c[1], self.c[6], self.calpha):
            t.grad = None
        score, _ = autograd.kernel_pool(self.c[0], self.c[1], self.c[2], self.c[3], self.c[4], self.c[5], self.c[6], self.calpha,
                                        self.log_scale)
        score.backward(self.gout)
        self.score = score.detach()   # detached: a kept autograd graph would break the CUDA-graph capture of the next step
        return self.c[0].grad

    def outputs(self, out):
        return {"scores": self.score, "grad_q": self.c[0].grad, "grad_d": self.c[1].grad, "grad_weight": self.c[6].grad,
                "grad_alpha": self.calpha.grad}

    def e2e_step(self):
        from matchmaker_b200 import autograd
        dq, dd, dqm, ddm = [t.to(self.dev, non_blocking=True) for t in self.h]
        dq.requires_grad_(True)
        dd.requires_grad_(True)
        score, _ = autograd.kernel_pool(dq, dd, dqm, ddm, self.c[4], self.c[5], self.c[6].detach(), self.calpha.detach(), self.log_scale)
        score.backward(self.gout)
        return torch.cat([score.detach().cpu(), dq.grad.sum().view(1).cpu()])

    e2e_note = "pinned host embeddings+masks -> H2D -> forward + backward kernels -> D2H scores (+ a gradient checksum)"

    def cpu_prepare(self):
        self.cpu_n = 64

    def cpu_step(self):
        from oracle import interaction_oracle as O
        n = self.cpu_n
        q = self.q[:n].clone().requires_grad_(True)
        d = self.d[:n].clone().requires_grad_(True)
        s = O.kernel_pool_tk(q, d, self.qm[:n], self.dm[:n], self.mu, self.sigma, self.alpha, self.w)[0]
        s.sum().backward()
        return q.grad


class TklWorkload:
    """BASELINE config 5: TKL interaction + window pooling, Lq=40, Ld=2000, D=300, 11 kernels, 16 docs per GPU
    (128 over 8 GPUs); op-level inputs = contextualised query + packed contextualised chunks."""
    bound = "hbm"
    dtype = "f32"
    name = "tkl_window_pool"
    metric = "query-doc pairs scored/sec (TKL chunked kernel pooling + window selection, Ld=2000)"
    kernel = "tkl_ts_kernel"
    launches_per_step = 4   # slot map, tile plan, window scores (tcgen05), top hills

    def __init__(self, rank, dev, B=128):
        from matchmaker_b200 import synthetic as O
        from matchmaker_b200.rankers.tkl import chunk_documents
        self.dev, self.B, self.Lq, self.Ld, self.D = dev, B, 40, 2000, 300
        g = torch.Generator().manual_seed(SEED + 20 + rank)
        self.q = torch.randn(B, self.Lq, self.D, generator=g) * 0.4
        d = torch.randn(B, self.Ld, self.D, generator=g) * 0.4
        q_len = torch.randint(3, self.Lq + 1, (B,), generator=g)
        d_len = O.synth_lengths(B, 1100.0, 500.0, 100, self.Ld, g)
        self.qm = (torch.arange(self.Lq).unsqueeze(0) < q_len.unsqueeze(1)).float()
        dm = (torch.arange(self.Ld).unsqueeze(0) < d_len.unsqueeze(1)).float()
        self.q = self.q * self.qm.unsqueeze(-1)
        d = d * dm.unsqueeze(-1)
        cd2, cp2, self.packed, self.pieces = chunk_documents(d, dm)
        self.chunks = cd2[self.packed][:, 5:-5].contiguous()   # overlap removed (sigir20_tkl.py:174)
        self.cmask = cp2[self.packed][:, 5:-5].contiguous()
        K = 11
        self.params = {"mu": torch.tensor([1.0, 0.9, 0.7, 0.5, 0.3, 0.1, -0.1, -0.3, -0.5, -0.7, -0.9]),
                       "sigma": torch.full((K,), 0.1), "dense_weight": torch.linspace(-0.014, 0.014, K),
                       "chunk_scoring": torch.ones(15), "sat_emb_reduce1_weight": torch.randn(self.D, generator=g) * 0.05,
                       "sat_normer_weight": torch.ones(2), "sat_normer_bias": torch.zeros(2),
                       "saturation_linear_weight": torch.tensor([0.01, -0.01]), "saturation_linear_bias": torch.tensor([100.0]),
                       "saturation_linear2_weight": torch.tensor([0.005, 0.01]), "saturation_linear2_bias": torch.tensor([100.0]),
                       "saturation_linear3_weight": torch.tensor([-0.01, 0.005]), "saturation_linear3_bias": torch.tensor([100.0])}
        p = self.params
        self.sat = torch.cat([p["sat_normer_weight"], p["sat_normer_bias"], p["saturation_linear_weight"],
                              p["saturation_linear_bias"], p["saturation_linear2_weight"], p["saturation_linear2_bias"],
                              p["saturation_linear3_weight"], p["saturation_linear3_bias"]])
        self.pairs = B
        per_pair = self.Lq * self.D * 4 + self.Ld * self.D * 4 + 8160
        self.alg_bytes = int(self.Lq * self.D * 4 * B + self.chunks.numel() * 4 + self.cmask.numel() * 4)
        self.alg_note = ("actual packed bytes: query + packed chunks + chunk masks (SURVEY 8(d) dense figure: %d "
                         "B/pair; documents here average %.0f of 2000 tokens)" % (per_pair, d_len.float().mean().item()))

    def to_device(self):
        d = self.dev
        p = self.params
        self.c = dict(q=self.q.to(d), qm=self.qm.to(d), ch=self.chunks.to(d), cm=self.cmask.to(d), pk=self.packed.to(d),
                      mu=p["mu"].to(d), sg=p["sigma"].to(d), dw=p["dense_weight"].to(d), sat=self.sat.to(d),
                      red=p["sat_emb_reduce1_weight"].to(d), cs=p["chunk_scoring"].to(d))

    def _run(self, q, qm, ch, cm, pk):
        from matchmaker_b200 import interaction
        c = self.c
        ws = interaction.tkl_window_scores(q, qm, ch, cm, pk, self.pieces, c["mu"], c["sg"], c["dw"], "embedding", c["sat"], c["red"])
        return interaction.tkl_top_hills(ws, c["cs"])[0]

    def kernel_step(self):
        c = self.c
        return self._run(c["q"], c["qm"], c["ch"], c["cm"], c["pk"])

    def outputs(self, out):
        return {"scores": out}

    def exchange(self, s):
        return s

    def pin(self):
        self.h = [t.pin_memory() for t in (self.q, self.qm, self.chunks, self.cmask, self.packed)]
        return sum(x.numel() * x.element_size() for x in self.h)

    def e2e_step(self):
        dv = [t.to(self.dev, non_blocking=True) for t in self.h]
        return self._run(*dv).cpu()

    e2e_note = "pinned host contextualised query/chunks -> H2D -> tkl_window_scores + tkl_top_hills -> D2H scores"

    def cpu_prepare(self):
        self.cpu_n = 8

    def cpu_step(self):
        from oracle import interaction_oracle as O
        n = self.cpu_n
        C = self.pieces
        pk = self.packed[:n * C]
        nc = int(pk.sum())
        with torch.no_grad():
            return O.tkl_interaction(self.q[:n], self.qm[:n], self.chunks[:nc], self.cmask[:nc], pk, C, self.params, "embedding")[0]

    def config(self, n_gpus):
        return {"workload": self.name, "docs_per_gpu": self.B, "Lq": self.Lq, "Ld": self.Ld, "dim": self.D, "kernels": 11,
                "saturation": "embedding", "pairs_per_step": self.B * n_gpus, "sharding": "documents split over ranks",
                "l2_policy": "inputs larger than L2 (%.2f GB per GPU per step)" % (self.alg_bytes / 1e9)}


class BertDotWorkload:
    """BASELINE config 4: BERT_DOT retrieval scoring, dim=768, 6400 queries x 8.8 M passages over 8 GPUs = 1.1 M
    passages per GPU (fp16, 1.69 GB), top-100; tensor-core bound."""
    bound = "tensor"
    dtype = "f16"
    name = "bert_dot_flat_ip_topk"
    metric = "query-passage pairs scored/sec (BERT_DOT exact inner-product top-100, dim=768)"
    kernel = "flat_ip_tc_kernel"
    launches_per_step = 3   # threshold fill, GEMM + top-k, merge

    def __init__(self, rank, dev, nq=6400, n_pass=1100000, k=100):
        from matchmaker_b200 import synthetic as O
        self.dev, self.nq, self.n, self.k, self.dim = dev, nq, n_pass, k, 768
        self.q, self.p = O.synth_dense_inputs(nq, n_pass, self.dim, seed=SEED + 30, shard_id=rank)
        self.pairs = nq * n_pass
        self.flops = 2.0 * nq * n_pass * self.dim
        self.alg_bytes = n_pass * self.dim * 2 + nq * self.dim * 2
        self.alg_note = "2*dim FLOP per (query, passage) pair; passages read once (1 536 B each)"
        self.id_base = rank * n_pass

    def to_device(self):
        self.cq, self.cp = self.q.to(self.dev), self.p.to(self.dev)

    def kernel_step(self):
        from matchmaker_b200 import interaction
        return interaction.flat_ip_topk(self.cq, self.cp, self.k, id_base=self.id_base)

    def outputs(self, out):
        return {"scores": out[0], "ids": out[1]}

    def exchange(self, si):
        from matchmaker_b200 import sharding
        return sharding.all_gather_merge(si[0], si[1], self.k)

    def pin(self):
        self.h = [self.q.pin_memory()]
        return self.h[0].numel() * 2

    def e2e_step(self):
        # the index (passages) is resident, as in FaissIdIndexer; per step the QUERIES travel (dense_retrieval.py:386-391)
        from matchmaker_b200 import interaction
        dq = self.h[0].to(self.dev, non_blocking=True)
        s, i = interaction.flat_ip_topk(dq, self.cp, self.k, id_base=self.id_base)
        return torch.cat([s.cpu().view(-1), i.cpu().view(-1).float()])

    e2e_note = "index resident in HBM (as faiss); pinned host queries -> H2D -> fused GEMM+top-k -> D2H (scores, ids)"

    def cpu_prepare(self):
        self.cq32, self.cpn = self.q[:64].float(), 200000  # 64-query x 200 k-passage slab (BASELINE.md section 2)

    def cpu_step(self):
        with torch.no_grad():
            s = self.cq32 @ self.p[:self.cpn].float().T
            return torch.topk(s, self.k, dim=1)

    def cpu_pairs(self):
        return 64 * self.cpn

    def config(self, n_gpus):
        return {"workload": self.name, "queries": self.nq, "passages_per_gpu": self.n, "dim": self.dim, "top_k": self.k,
                "storage_dtype": "float16", "pairs_per_step": self.pairs * n_gpus,
                "sharding": "passages sharded over ranks; per-query top-k all-gather + merge when N>1",
                "l2_policy": "passage shard 1.69 GB per GPU, larger than L2"}


WORKLOADS = ["colbert", "tk", "knrm", "tkl", "bert_dot", "tk_train"]
SECONDARY = ["tk", "knrm", "tkl", "bert_dot", "tk_train"]


def make_workload(name, rank, dev):
    if name == "colbert":
        return ColbertWorkload(rank, dev)
    if name in ("tk", "knrm"):
        return KernelPoolWorkload(rank, dev, name)
    if name == "tk_train":
        return KernelPoolTrainWorkload(rank, dev)
    if name == "tkl":
        return TklWorkload(rank, dev)
    if name == "bert_dot":
        return BertDotWorkload(rank, dev)
    raise SystemExit("unknown workload " + name)


def _cpu_threads():
    """Threads for the CPU legs.  torchrun exports OMP_NUM_THREADS=1 to its workers, which would throttle the reference
    arm to one core for N > 1 (round 1: 38.8 k pairs/s at N=2 against 957 k at N=1 on the same box); the CPU arm
    always asks for every physical core explicitly (MMB200_REF_THREADS overrides)."""
    env = os.environ.get("MMB200_REF_THREADS")
    if env:
        return max(1, int(env))
    try:
        import psutil
        n = psutil.cpu_count(logical=False) or 0
    except Exception:  # noqa: BLE001
        n = 0
    if n <= 0:
        n = max(1, (os.cpu_count() or 2) // 2)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


def _cpu_per_step(wl):
    return wl.cpu_pairs() if hasattr(wl, "cpu_pairs") else (getattr(wl, "cpu_n", None) or wl.pairs)


def time_cpu(wl, budget_s=12.0, max_reps=50, one_thread_budget_s=4.0):
    """cpu_baseline: the oracle port of the reference's PyTorch path on this host's cores (all physical cores), plus the
    same step on ONE thread -- the reference's own runner setting (train.py:12 pins OMP_NUM_THREADS=1)."""
    prev = torch.get_num_threads()
    torch.set_num_threads(_cpu_threads())
    wl.cpu_prepare()
    wl.cpu_step()  # warm-up
    reps, t_total = 0, 0.0
    while t_total < budget_s and reps < max_reps:
        t0 = time.perf_counter()
        wl.cpu_step()
        t_total += time.perf_counter() - t0
        reps += 1
    per = _cpu_per_step(wl)
    out = {"value": per * reps / t_total, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
           "sample": "%d x %d pairs of this workload through the oracle (torch CPU fp32, %d threads of %d logical cores)"
                     % (reps, per, torch.get_num_threads(), os.cpu_count())}
    if one_thread_budget_s > 0:
        torch.set_num_threads(1)
        t0 = time.perf_counter()
        wl.cpu_step()
        dt = time.perf_counter() - t0
        n1 = 1
        while dt < one_thread_budget_s and n1 < 5:
            t1 = time.perf_counter()
            wl.cpu_step()
            dt += time.perf_counter() - t1
            n1 += 1
        out["one_thread"] = {"value": per * n1 / dt, "unit": "pairs/s", "cores": 1,
                             "note": "same step with torch.set_num_threads(1) (the reference runner's OMP_NUM_THREADS=1, train.py:12)"}
    torch.set_num_threads(prev)
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU PyTorch path (oracle port) on this host, rank 0 only.  `config` is the GPU
    arm's config at N=1 verbatim; what one CPU step covers is said in `cpu_baseline.sample`."""
    if rank != 0:
        return
    torch.set_num_threads(_cpu_threads())
    wl = make_workload(args.workload, 0, torch.device("cpu"))
    wl.cpu_prepare()
    for _ in range(args.warmup):
        wl.cpu_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        wl.cpu_step()
    dt = time.perf_counter() - t0
    per = _cpu_per_step(wl)
    v = per * args.steps / dt
    line = {"impl": "reference", "metric": wl.metric, "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": wl.config(1),
            "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "each step = %d pairs of the workload on %d torch threads (%d logical cores); "
                                       "under torchrun rank 0 alone runs it" % (per, torch.get_num_threads(), os.cpu_count())},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _roofline(wl, kern_ms, workload_key):
    hbm_peak, peak_src = _peaks()
    if wl.bound == "hbm":
        achieved = wl.alg_bytes / (kern_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": wl.kernel, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": None, "peak_source": peak_src, "kernel_ms": kern_ms,
                "algorithmic_bytes_per_launch": wl.alg_bytes, "algorithmic_bytes": wl.alg_note}
    else:
        tf_peak, tf_src = _tensor_peak()
        achieved = wl.flops / (kern_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": wl.kernel, "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s",
                "frac": achieved / tf_peak, "traffic": None, "peak_source": tf_src, "kernel_ms": kern_ms,
                "algorithmic_flops_per_launch": wl.flops, "algorithmic_flops": wl.alg_note}
    # DRAM bytes per launch of the dominant kernel: NOT measured in this run (ncu cannot run inside a timed bench) --
    # copied from the committed `ncu --set full` capture of this workload under profiles/
    prof = os.path.join(ROOT, "profiles", "maxsim_traffic.json" if workload_key == "colbert" else f"{workload_key}_traffic.json")
    if os.path.isfile(prof):
        try:
            j = json.load(open(prof))
            roof["traffic"] = j["dram_bytes_per_launch"]
            roof["traffic_source"] = "static ncu capture (%s, %s)" % (os.path.relpath(prof, ROOT), j.get("capture", "profiles/"))
        except Exception:  # noqa: BLE001
            pass
    return roof


def graphed_step(fn, dev):
    """Capture one step (a handful of short launches: with a Python caller the host issues them more slowly than the GPU
    retires them) into a CUDA graph and return a replay closure; None if the step cannot be captured.  The kernels, their
    arguments and their order are those of the eager step; only the launch path changes."""
    try:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn()
        g.replay()
        torch.cuda.synchronize(dev)

        def replay():
            g.replay()
            return out
        return replay
    except Exception as e:  # noqa: BLE001
        sys.stderr.write("bench: CUDA-graph capture of the step failed (%r); running it eagerly\n" % (e,))
        try:
            torch.cuda.synchronize(dev)
        except Exception:  # noqa: BLE001
            pass
        return None


def bench_secondary(name, dev, steps, cpu_budget_s):
    """One sub-record per secondary BASELINE config, measured inside the default run at N=1 so that the driver's run
    times every workload, not only the headline one: value (HBM-resident, CUDA events), roofline, e2e, CPU port."""
    wl = make_workload(name, 0, dev)
    wl.to_device()
    for _ in range(3):
        wl.kernel_step()
    torch.cuda.synchronize()
    step = graphed_step(wl.kernel_step, dev) if (wl.launches_per_step > 1 and getattr(wl, "graph_ok", True)) else None
    graphed = step is not None
    step = step or wl.kernel_step
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    h2d = wl.pin()
    wl.e2e_step()
    torch.cuda.synchronize()
    n_e2e = 5   # each step ends in a device->host read: per-step wall times, median (one slow step -- first touch of the
    walls = []  # pinned pages, an allocator trim -- moved a two-step mean by 9x between otherwise identical runs)
    for _ in range(n_e2e):
        t0 = time.perf_counter()
        out = wl.e2e_step()
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    e2e_s = sorted(walls)[n_e2e // 2]
    rec = {"metric": wl.metric, "value": wl.pairs / (ms * 1e-3), "unit": "pairs/s", "steps": steps, "ms_per_step": ms,
           "dtype": wl.dtype, "config": dict(wl.config(1), cuda_graph=graphed), "roofline": _roofline(wl, ms, name),
           "gpu_launches": steps * wl.launches_per_step,
           "e2e": {"value": wl.pairs / e2e_s, "unit": "pairs/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": out.numel() * out.element_size(), "ms_per_step": e2e_s * 1e3,
                   "steps": n_e2e, "statistic": "median of per-step wall times", "note": wl.e2e_note}}
    if cpu_budget_s > 0:
        rec["cpu_baseline"] = time_cpu(wl, budget_s=cpu_budget_s, max_reps=10, one_thread_budget_s=0)
    if name == "tkl":
        # the same step on four times as many documents: the three helper kernels around tkl_ts_kernel (slot map, tile plan,
        # top hills: ~25 us, latency-bound, independent of the batch) weigh a quarter as much -- next to the 128-document
        # figure, not instead of it
        del wl
        torch.cuda.empty_cache()
        big = TklWorkload(0, dev, B=512)
        big.to_device()
        for _ in range(3):
            big.kernel_step()
        torch.cuda.synchronize()
        bstep = graphed_step(big.kernel_step, dev) or big.kernel_step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            bstep()
        e1.record()
        torch.cuda.synchronize()
        bms = e0.elapsed_time(e1) / steps
        rec["at_512_docs"] = {"value": big.pairs / (bms * 1e-3), "unit": "pairs/s", "ms_per_step": bms,
                              "roofline_frac": _roofline(big, bms, name)["frac"]}
    if name == "tk_train":
        # the same step at the forward workload's batch (4096 pairs, 28 per SM instead of 7): the persistent kernels'
        # prologue and the pair boundaries weigh less -- reported next to the 1024-pair figure, not instead of it
        del wl
        torch.cuda.empty_cache()
        big = KernelPoolTrainWorkload(0, dev, pairs=4096)
        big.to_device()
        for _ in range(3):
            big.kernel_step()
        torch.cuda.synchronize()
        bstep = graphed_step(big.kernel_step, dev) or big.kernel_step
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            bstep()
        e1.record()
        torch.cuda.synchronize()
        bms = e0.elapsed_time(e1) / steps
        rec["at_4096_pairs"] = {"value": big.pairs / (bms * 1e-3), "unit": "pairs/s", "ms_per_step": bms,
                                "roofline_frac": _roofline(big, bms, name)["frac"]}
    return rec


DUMP_SAMPLE = 1 << 22          # elements kept of a larger output (16 MB in float32)
DUMP_LIMIT = 64 << 20          # bytes written by --dump-outputs in all


def dump_outputs(out_dir, arrays):
    """Write each output of the last timed step as out_dir/<name>.npy: floating-point outputs as float32, integer ones
    (ids) as float64, which holds them exactly.  An output of more than DUMP_SAMPLE elements is written as the same
    seeded sample of its flattened elements on every run, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(SEED))[:DUMP_SAMPLE].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.cpu().numpy().astype(np.float32 if t.is_floating_point() else np.float64)
        total += a.nbytes
        assert total <= DUMP_LIMIT, "--dump-outputs: more than %d bytes" % DUMP_LIMIT
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="colbert", choices=WORKLOADS)
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed end-to-end steps (default: min(steps, 5))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="never replay the step from a CUDA graph")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the per-workload sub-records (tk, knrm, tkl, bert_dot, ...) of the default N=1 run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what rank 0's last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    wl = make_workload(args.workload, rank, dev)
    wl.to_device()

    # N > 1: scoring runs on a HIGH-priority stream, the top-k exchange on a normal-priority side stream.  The scoring
    # kernels are persistent (one CTA per SM, nearly all of its shared memory); if the exchange's kernels (top-k, NCCL
    # all-gather, merge) win SMs first, the displaced CTAs start late and -- NCCL kernels spin until every rank has
    # arrived -- the ranks convoy (measured at N = 4: 1.2 ms per step for a 0.52 ms kernel).  With priorities the block
    # scheduler places the next step's CTAs first and the exchange fills in behind them.
    side = torch.cuda.Stream() if world > 1 else None
    if world > 1:
        torch.cuda.synchronize()   # the uploads above ran on the default stream
        torch.cuda.set_stream(torch.cuda.Stream(priority=-1))

    def exchange_async(out):
        """The top-k exchange of step i runs on a side stream and overlaps the scoring kernel of step i+1 (a
        serving loop would do the same); the timed region ends only after every exchange has finished."""
        ev = torch.cuda.Event()
        ev.record()
        with torch.cuda.stream(side):
            side.wait_event(ev)
            for t_ in (out if isinstance(out, (tuple, list)) else (out,)):
                t_.record_stream(side)
            return wl.exchange(out)

    def step():
        out = wl.kernel_step()
        return exchange_async(out) if world > 1 else out

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    if world > 1:
        torch.cuda.current_stream().wait_stream(side)
    sync_all()
    kstep = wl.kernel_step
    graphed = False
    if world == 1 and wl.launches_per_step > 1 and getattr(wl, "graph_ok", True) and not args.no_graph:
        g = graphed_step(wl.kernel_step, dev)
        if g is not None:
            kstep, graphed = g, True

    # ---- timed region: `value` (inputs resident in HBM) -----------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    kern_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    t_val0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        kern_ev[i][0].record()
        out = kstep()
        kern_ev[i][1].record()
        if world > 1:
            exchange_async(out)
    if world > 1:
        torch.cuda.current_stream().wait_stream(side)
    e1.record()
    sync_all()
    t_val1 = time.perf_counter()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl.outputs(out))
    ms_total = e0.elapsed_time(e1)
    kern_ms = statistics.mean(a.elapsed_time(b) for a, b in kern_ev)
    t = torch.tensor([ms_total, kern_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kern_ms = t.tolist()
    ms_per_step = ms_total / args.steps
    pairs_per_step = wl.pairs * world
    value = pairs_per_step / (ms_per_step * 1e-3)

    # ---- e2e: public API with HOST buffers, H2D + kernel + D2H inside the timed region -------------
    h2d = wl.pin()
    e2e_steps = args.e2e_steps or min(args.steps, 5)
    for _ in range(2):
        wl.e2e_step()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out = wl.e2e_step()  # ends with a device->host read of the result
    torch.cuda.synchronize()
    t_e2e1 = time.perf_counter()
    clocks = sampler.stop([(t_val0, t_val1), (t0, t_e2e1)]) if rank == 0 else None
    e2e_s = (t_e2e1 - t0) / e2e_steps
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = te.item()
    d2h = out.numel() * out.element_size()

    if rank == 0:
        line = {"metric": wl.metric, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic", "config": dict(wl.config(world), cuda_graph=graphed),
                "clocks": clocks,
                "e2e": {"value": pairs_per_step / e2e_s, "unit": "pairs/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s * 1e3, "note": wl.e2e_note},
                "gpu_launches": args.steps * wl.launches_per_step,
                "roofline": _roofline(wl, kern_ms, args.workload)}
        if hasattr(wl, "h2d_dense"):
            line["e2e"]["h2d_bytes_dense"] = wl.h2d_dense
        if args.workload == "colbert":
            # informational: same workload with the ragged fetch (padding rows are never read from HBM)
            from matchmaker_b200 import interaction
            for _ in range(3):
                interaction.maxsim(wl.cq, wl.cd, wl.cqm, wl.cdm, docs_per_query=DOCS_PER_QUERY, impl="tcgen05_ragged")
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            for _ in range(args.steps):
                interaction.maxsim(wl.cq, wl.cd, wl.cqm, wl.cdm, docs_per_query=DOCS_PER_QUERY, impl="tcgen05_ragged")
            r1.record()
            torch.cuda.synchronize()
            line["skip_padding"] = {"value": wl.pairs * args.steps / (r0.elapsed_time(r1) * 1e-3), "unit": "pairs/s",
                                    "note": "impl=tcgen05_ragged on the same HBM-resident inputs, 1 GPU: rows past each "
                                            "document's last unmasked token are not fetched (mean 75 of 180 tokens); not "
                                            "used for `value` or the roofline"}
            if world == 1:
                # the same public call for a caller that does NOT pin: pageable host tensors, staged slab pipeline
                wl.e2e_pageable_step()
                tp = time.perf_counter()
                wl.e2e_pageable_step()
                tp = time.perf_counter() - tp
                line["e2e"]["pageable"] = {"value": wl.pairs / tp, "unit": "pairs/s", "ms_per_step": tp * 1e3,
                                           "h2d_bytes_per_step": wl.h2d_dense,
                                           "note": "same call on pageable host tensors: nothing is pinned anywhere, the library "
                                                   "stages 96 MB slabs (cudaMemcpyAsync from pageable memory), every padded row travels"}
                del wl.pg
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = time_cpu(wl)
        if world == 1 and args.workload == "colbert" and not args.no_secondary:
            # free the headline workload's 3 GB before the secondary ones allocate theirs
            for a in ("cd", "cdm", "d", "dm", "h", "q32", "d32"):
                if hasattr(wl, a):
                    delattr(wl, a)
            torch.cuda.empty_cache()
            subs = {}
            for name in SECONDARY:
                try:
                    subs[name] = bench_secondary(name, dev, steps=min(args.steps, 10), cpu_budget_s=0 if args.no_cpu_baseline else 3.0)
                except Exception as e:  # noqa: BLE001  (a failing secondary workload must not lose the headline line)
                    subs[name] = {"error": repr(e)}
                torch.cuda.empty_cache()
            line["workloads"] = subs
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
