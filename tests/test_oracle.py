"""CPU suite, part 1: the oracle restatement against the committed golden vectors (made by the
reference's own classes under oracle/shim) and -- when /root/reference is mounted -- against the
reference run live.  Bar: bit-exact (max |diff| == 0.0), same dtype as the reference script."""
import numpy as np
import pytest
import torch

from conftest import Golden, golden_cases
from oracle import ref_loader, restate

pytestmark = pytest.mark.usefixtures("one_cpu_thread")


@pytest.mark.parametrize("name", golden_cases())
def test_restatement_matches_golden_bit_exact(name):
    g = Golden(name)
    out = restate.decode(g.program, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=g.dtype)
    assert out["prob"].dtype == g.dtype
    assert torch.equal(out["prob"], g.prob)
    # prob == sigmoid(-logit) (classical programs additionally clamp)
    p = torch.sigmoid(-out["logit"])
    if g.program in ("cgnni", "bp_classical"):
        p = p.clamp(1e-7, 1 - 1e-7)
    assert torch.equal(p, g.prob)


@pytest.mark.parametrize("name", golden_cases())
def test_single_phase_matches_golden_bit_exact(name):
    g = Golden(name)
    for phase, want in (("var", g.phase_var), ("chk", g.phase_chk)):
        got = restate.propagate(g.program, phase, g.edge_index, g.V, g.C, g.m0, g.x, g.weights, dtype=g.dtype)
        assert torch.equal(got, want), phase


def test_edge_order_is_row_major_coo():
    # H.to_sparse()._indices() is sorted by variable then check (decoder_v2_4.py:164-165)
    for name in golden_cases():
        g = Golden(name)
        v, c = np.nonzero(g.H.numpy())
        assert np.array_equal(np.stack([v, c]), g.edge_index.numpy())


def test_empty_batch():
    g = Golden("cgnni_ldpc_epoch18")
    out = restate.decode(g.program, g.edge_index, g.V, g.C, g.x[:0], g.weights, T=2)
    assert out["prob"].shape == (0, g.V)


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not mounted")
def test_restatement_matches_live_reference():
    """Re-run the reference's own GNNI under the shim on fresh seeded inputs (different seed and
    batch size from the fixtures) and compare bit for bit."""
    with ref_loader.reference_session("quantum"):
        ns = ref_loader.load_reference("quantum/decoder_v2_4.py",
                                       consts={"BATCH_SIZE": "6", "run1": "6", "run2": "6", "L": "4"}, seed=99)
        dec = ns.GNNI(3)
        dec.load_state_dict(torch.load(ref_loader.REF_ROOT + "/quantum/new_model/decoder_parameters_epoch2.pkl"))
        batch = next(iter(ns.train_loader))
        with torch.no_grad():
            want = dec(batch)
        rows, cols = int(ns.rows), int(ns.cols)
        ei = batch.edge_index[:, : batch.edge_index.size(1) // 6]
        got = restate.decode("v2_4", ei, rows, cols, batch.x.reshape(6, rows + cols), dec.state_dict(), T=3)
    assert torch.equal(got["prob"].reshape(-1, 1), want)
