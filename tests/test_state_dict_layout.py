"""Checkpoint compatibility: the drop-in rankers expose exactly the state-dict keys and shapes of the reference's
classes (fixture recorded from the reference by oracle/make_state_dict_fixture.py).  The reference loads checkpoints
with load_state_dict(strict=False) (train.py:107, dense_retrieval.py:138), which silently skips mismatching keys -- a
renamed parameter would train from scratch without an error."""
import json
import os

import pytest
import torch

from conftest import ROOT
from matchmaker_b200.rankers import ECAI20_TK, KNRM
from matchmaker_b200.rankers.tkl import TKL_sigir20
from oracle import interaction_oracle as O

LAYOUT = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_layout.json")))
MU11, SG11 = O.knrm_kernel_mus(11), O.knrm_kernel_sigmas(11)
MU21, SG21 = O.tk_21_kernels()


def _layout(module):
    return {k: list(v.shape) for k, v in module.state_dict().items()}


CASES = {
    "knrm_11": lambda: KNRM(11),
    "tk_emb300_k11_len200": lambda: ECAI20_TK(300, MU11, SG11, 10, 2, 300, 200, True, True),
    "tk_emb300_k21_len200": lambda: ECAI20_TK(300, MU21, SG21, 10, 2, 300, 200, True, True),
    "tkl_emb300_k11_len2000_embedding": lambda: TKL_sigir20(300, MU11, SG11, 10, 2, 300, 2000, True, True, "embedding"),
    "tkl_emb300_k11_len2000_log": lambda: TKL_sigir20(300, MU11, SG11, 10, 2, 300, 2000, True, True, "log"),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_state_dict_keys_and_shapes_match_the_reference(name):
    ours, ref = _layout(CASES[name]()), LAYOUT[name]
    assert sorted(ours) == sorted(ref), (f"missing: {sorted(set(ref) - set(ours))}, unexpected: {sorted(set(ours) - set(ref))}")
    for k in ref:
        assert ours[k] == ref[k], f"{name}: {k} has shape {ours[k]}, the reference has {ref[k]}"


def test_reference_checkpoint_round_trip():
    """A state dict with the reference's layout loads strictly, and the parameters the kernels read come out intact."""
    m = CASES["tk_emb300_k21_len200"]()
    g = torch.Generator().manual_seed(3)
    sd = {k: torch.randn(shape, generator=g) for k, shape in LAYOUT["tk_emb300_k21_len200"].items()}
    missing, unexpected = m.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    assert torch.equal(m.kernel_bin_weights.weight, sd["kernel_bin_weights.weight"])
    assert torch.equal(m.kernel_alpha_scaler, sd["kernel_alpha_scaler"])
    assert torch.equal(m.mu, sd["mu"]) and torch.equal(m.sigma, sd["sigma"])


def test_fixture_regenerates_from_the_reference():
    """A separate recording of the reference's layouts (tests/golden/state_dict_layout_regen.json,
    `python -m oracle.make_state_dict_fixture regen`) agrees with the fixture."""
    regen = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_layout_regen.json")))
    assert regen["knrm_11"] == LAYOUT["knrm_11"]
    assert regen["tk_emb300_k21_len200"] == LAYOUT["tk_emb300_k21_len200"]
    assert regen["tkl_emb300_k11_len2000_log"] == LAYOUT["tkl_emb300_k11_len2000_log"]


def test_from_config_reads_the_reference_keys():
    """`config["model"]` strings and the config keys each `from_config` reads (models/all.py:141-184, knrm.py:21-22,
    ecai20_tk.py:22-32, sigir20_tkl.py:17-29): a config written for the reference builds the same module here."""
    from matchmaker_b200.rankers import get_model_class
    cfg = {"knrm_kernels": 11, "tk_kernels_mu": MU21, "tk_kernels_sigma": SG21, "tk_att_heads": 10, "tk_att_layer": 2,
           "tk_att_ff_dim": 300, "max_doc_length": 200, "tk_use_diff_posencoding": True, "tk_mix_hybrid_context": True,
           "tk_use_pos_encoding": True, "tk_saturation_type": "embedding"}
    assert _layout(get_model_class("knrm").from_config(cfg, 300)) == LAYOUT["knrm_11"]
    assert _layout(get_model_class("TK").from_config(cfg, 300)) == LAYOUT["tk_emb300_k21_len200"]
    cfg_tkl = dict(cfg, tk_kernels_mu=MU11, tk_kernels_sigma=SG11, max_doc_length=2000)
    assert _layout(get_model_class("TKL").from_config(cfg_tkl, 300)) == LAYOUT["tkl_emb300_k11_len2000_embedding"]
    with pytest.raises(KeyError):
        get_model_class("matchpyramid")   # outside the hot path: fails loudly instead of silently substituting
    # the kernel-pooling variants of SURVEY 8(f) read the reference's keys too (conv_knrm.py:20-25, cikm20_tk_sparse.py:19-29)
    ck = get_model_class("conv_knrm").from_config({"conv_knrm_ngrams": 3, "conv_knrm_kernels": 11, "conv_knrm_conv_out_dim": 128}, 300)
    assert ck.dense.weight.shape == (1, 99) and len(ck.convolutions) == 3
    ts = get_model_class("TK_Sparse").from_config(dict(cfg, tk_att_proj_dim=32), 300)
    assert {"mixer_stop", "stop_word_reducer.weight", "stop_word_reducer2.bias", "kernel_alpha_scaler"} <= set(ts.state_dict().keys())
