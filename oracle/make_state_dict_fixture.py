"""Test infrastructure (not product code): record the state-dict layout of the reference's non-BERT rankers.

Instantiates KNRM / ECAI20_TK / TKL_sigir20 from /root/reference through oracle/reference_loader.py (allennlp / CUDA
constructor shims) and writes {model: {key: [shape], ...}} to tests/golden/state_dict_layout.json.  A checkpoint written
by the reference loads into the drop-in classes iff these keys and shapes match (train.py:107 and
dense_retrieval.py:138 call load_state_dict(strict=False), which silently SKIPS keys that do not match).

    python -m oracle.make_state_dict_fixture [regen]

`regen` records three of those layouts a second time into tests/golden/state_dict_layout_regen.json, which
tests/test_state_dict_layout.py checks the fixture against without needing the reference sources.
"""
import json
import os
import sys

from oracle import reference_loader as R
from oracle import interaction_oracle as S

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
OUT = os.path.join(GOLDEN, "state_dict_layout.json")
REGEN_OUT = os.path.join(GOLDEN, "state_dict_layout_regen.json")


def layout(module):
    return {k: list(v.shape) for k, v in module.state_dict().items()}


def main(path=OUT, keys=None):
    mu11, sg11 = S.knrm_kernel_mus(11), S.knrm_kernel_sigmas(11)
    mu21, sg21 = S.tk_21_kernels()
    out = {
        "knrm_11": layout(R.load_knrm(11)),
        "tk_emb300_k11_len200": layout(R.load_tk(300, mu11, sg11, 10, 2, 300, 200, True, True)),
        "tk_emb300_k21_len200": layout(R.load_tk(300, mu21, sg21, 10, 2, 300, 200, True, True)),
        "tkl_emb300_k11_len2000_embedding": layout(R.load_tkl(300, mu11, sg11, 10, 2, 300, 2000, True, True, "embedding")),
        "tkl_emb300_k11_len2000_log": layout(R.load_tkl(300, mu11, sg11, 10, 2, 300, 2000, True, True, "log")),
    }
    if keys:
        out = {k: out[k] for k in keys}
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    for k, v in out.items():
        print(k, len(v), "tensors")


if __name__ == "__main__":
    if sys.argv[1:] == ["regen"]:
        main(REGEN_OUT, ["knrm_11", "tk_emb300_k21_len200", "tkl_emb300_k11_len2000_log"])
    else:
        main()
