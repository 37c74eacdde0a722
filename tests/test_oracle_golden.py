"""Pin oracle/mmsum_oracle.py (the CPU restatement) against golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py, run with a checkout of the reference present)."""
import pytest
import torch

from golden_util import compare_grads, load_golden
from oracle import mmsum_oracle as OR

SMALL = ["small_yelp", "small_yelp_gates_open", "small_amazon", "small_text", "small_img", "small_table_yelp", "small_table_amazon"]


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference_golden_small(name):
    gold = load_golden(name)
    loss, grads, _ = OR.step_loss_and_grads(gold["sd"], gold["cfg"], gold["batch"], gold["label_smoothing"],
                                            dtype=torch.float32)
    assert abs(loss.item() - gold["loss"]) <= 2e-6 * abs(gold["loss"])
    bad = compare_grads(gold, grads, rel_tol=2e-4)
    assert not bad, bad[:5]


def test_oracle_fp64_agrees_with_fp32_reference():
    # the fp64 oracle is the high-precision anchor the CUDA path is compared with at full size
    gold = load_golden("small_yelp_gates_open")
    loss, grads, _ = OR.step_loss_and_grads(gold["sd"], gold["cfg"], gold["batch"], 0.1, dtype=torch.float64)
    assert abs(loss.item() - gold["loss"]) <= 2e-6 * abs(gold["loss"])
    assert not compare_grads(gold, grads, rel_tol=2e-4)


@pytest.mark.slow
def test_oracle_matches_reference_golden_full_bart_large():
    gold = load_golden("full_yelp_b1")
    torch.set_num_threads(max(1, torch.get_num_threads()))
    loss, grads, _ = OR.step_loss_and_grads(gold["sd"], gold["cfg"], gold["batch"], 0.1, dtype=torch.float32)
    assert abs(loss.item() - gold["loss"]) <= 5e-6 * abs(gold["loss"])
    bad = compare_grads(gold, grads, rel_tol=1e-3)
    assert not bad, bad[:5]


def test_shift_tokens_right_cases():
    # the four documented cases of modeling_multimodalsum.py:225-246
    ids = torch.tensor([[5, 6, 7, 8, 2, 1, 1], [9, 10, 2, 1, 1, 1, 1]])
    out = OR.shift_tokens_right(ids, 1, 0, 2)
    assert out.tolist() == [[0, 5, 6, 7, 8, 1, 1], [0, 9, 10, 1, 1, 1, 1]]
    ids = torch.tensor([[0, 6, 7, 8, 2]])
    assert OR.shift_tokens_right(ids, 1, 0, 2).tolist() == [[2, 0, 6, 7, 8]]
