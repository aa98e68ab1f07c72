"""The CPU restatement of the ESANet guidance network (oracle/esanet.py) against the outputs of the reference's ESANetOneModality
on the same synthetic weights and inputs (tests/golden/esanet_*.npz).  No GPU needed."""
import numpy as np
import pytest
import torch


@pytest.mark.parametrize("name", ["r18_small", "r34_full"])
def test_oracle_esanet_against_reference(name, golden_dir):
    from make_esanet_golden import ESANET_CASES, esanet_input, esanet_weights
    from _synth import state_dict_digest
    from oracle.esanet import esanet_forward
    from rdfc_gan_b200.esanet import ESANetOneModality
    c = ESANET_CASES[name]
    gold = np.load(f"{golden_dir}/esanet_{name}.npz")
    sd = esanet_weights(ESANetOneModality(**c["kw"]).eval(), c["seed"])
    assert state_dict_digest(sd) == int(gold["digest"][0]), "synthetic weights differ from the ones the golden used"
    y = esanet_forward(sd, esanet_input(c))
    assert y.dtype == torch.float32 and y.shape[:2] == (c["B"], 40)
    got = y.numpy()[:, :, ::c["stride"], ::c["stride"]]
    assert got.shape == gold["logits"].shape
    # the same torch CPU calls as the reference in the same order: equal up to CPU fp32 summation-order noise
    assert float(np.abs(got - gold["logits"]).max()) <= 1e-5 * float(gold["rms"])
