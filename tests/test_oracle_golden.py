"""Pins the CPU oracle (oracle/) to the UNMODIFIED reference through the committed goldens
(tests/golden/*.npz, produced by tests/golden/make_golden.py from /root/reference)."""
import numpy as np
import pytest
import torch

from fira_testlib import golden_batch, load_batch_golden, load_model_golden, load_raw_golden, seeded_model

import fira_oracle as O
import graph_oracle as GO


@pytest.fixture(scope="module")
def sd():
    return {k: v.detach().clone() for k, v in seeded_model().state_dict().items()}


@pytest.fixture(scope="module")
def gold():
    return load_model_golden()


def test_position_table_matches_reference_formula():
    import math
    tab = O.position_table(30, 256)
    for i in (0, 1, 7, 29):
        for j in (0, 1, 63, 127):
            assert abs(tab[i, 2 * j].item() - math.sin(i / 10000 ** (2 * j / 256))) < 1e-6
            assert abs(tab[i, 2 * j + 1].item() - math.cos(i / 10000 ** (2 * j / 256))) < 1e-6


def test_graph_oracle_reproduces_reference_process_data():
    raw = load_raw_golden()
    g = load_batch_golden()
    ptr = g["edge_ptr"]
    for i in range(0, 128, 3):
        c = GO.build_commit(raw["raw"], i, raw["word_vocab"], raw["ast_change_vocab"], raw["VOCAB_UPPER_CASE"])
        for k in ("sou", "tar", "mark", "ast_change", "tar_label", "sub_token"):
            assert np.array_equal(np.array(c[k]), g[k][i]), (i, k)
        assert np.array_equal(np.array(c["attr"]), g["attr"][i]), (i, "attr")
        # same edge list in the same insertion order, bit-identical float64 values
        assert np.array_equal(np.array(c["row"]), g["edge_row"][ptr[i]:ptr[i + 1]])
        assert np.array_equal(np.array(c["col"]), g["edge_col"][ptr[i]:ptr[i + 1]])
        assert np.array_equal(np.array(c["val"]), g["edge_val"][ptr[i]:ptr[i + 1]])


def test_oracle_forward_matches_reference(sd, gold):
    torch.set_num_threads(8)
    with torch.no_grad():
        batch = golden_batch(0, 32)
        detail = {}
        loss_sum, n_tok = O.forward(sd, *batch, stage="train", detail=detail)
        ids = O.forward(sd, *batch, stage="dev")
    assert int(n_tok) == int(gold["mask_sums"][0])
    assert abs(loss_sum.item() - gold["loss_sums"][0]) <= 1e-4 * abs(gold["loss_sums"][0])
    np.testing.assert_allclose(detail["nll"].numpy(), gold["nll"][:32], rtol=1e-4, atol=1e-5)
    assert np.array_equal(ids.numpy(), gold["dev_ids"][:32])
    np.testing.assert_allclose(detail["memory"][:4, :, ::2].numpy(), gold["full_memory_even"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(detail["decoder"][:4].numpy(), gold["full_decoder"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(detail["logp"][:4].max(-1).values.numpy(), gold["full_logp_max"], rtol=1e-4, atol=1e-5)
    mem_abs = (detail["memory"].abs() * detail["mem_mask"].unsqueeze(-1)).sum((1, 2)).numpy()
    np.testing.assert_allclose(mem_abs, gold["mem_abs"][:32], rtol=1e-4)


def test_oracle_forward_matches_reference_on_edge_commits(sd):
    """DataSet extremes + crafted truncation commits (tests/golden/make_golden_edge.py): reference-built inputs,
    reference model outputs (model_edge.npz)."""
    import os
    from fira_testlib import GOLDEN, load_edge_golden
    _, g = load_edge_golden()
    ref = np.load(os.path.join(GOLDEN, "model_edge.npz"))
    n = len(g["sou"])
    t = lambda k: torch.from_numpy(g[k].astype(np.int64))
    ptr = g["edge_ptr"]
    dense = torch.stack([O.dense_adjacency(g["edge_row"][ptr[i]:ptr[i + 1]], g["edge_col"][ptr[i]:ptr[i + 1]],
                                           g["edge_val"][ptr[i]:ptr[i + 1]]) for i in range(n)])
    batch = [t("sou"), t("tar"), t("attr"), t("mark"), t("ast_change"), dense, t("tar_label"), t("sub_token")]
    torch.set_num_threads(8)
    with torch.no_grad():
        loss_sum, n_tok = O.forward(sd, *batch, stage="train")
        ids = O.forward(sd, *batch, stage="dev")
        one = [O.forward(sd, *[b[i:i + 1] for b in batch], stage="train")[0].item() for i in range(n)]
    assert int(n_tok) == int(ref["mask_sum"])
    assert abs(loss_sum.item() - float(ref["loss_sum"])) <= 1e-4 * float(ref["loss_sum"])
    np.testing.assert_allclose(np.array(one), ref["loss_per_commit"], rtol=1e-4)
    assert np.array_equal(ids.numpy(), ref["argmax_ids"])


def test_oracle_gradients_match_reference(sd, gold):
    torch.set_num_threads(8)
    n = int(gold["grad_commits"])
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss_sum, n_tok = O.forward(params, *golden_batch(0, n), stage="train")
    loss = loss_sum / n_tok
    loss.backward()
    assert abs(loss.item() - float(gold["grad_loss"])) < 1e-4 * float(gold["grad_loss"])
    keys = [str(k) for k in gold["grad_keys"]]
    with_grad = [k for k, p in params.items() if p.grad is not None]
    assert sorted(with_grad) == sorted(keys)          # same 264 tensors receive gradient
    for j, k in enumerate(keys):
        g = params[k].grad
        ref = gold["grad_norm"][j]
        assert abs(g.double().norm().item() - ref) <= 2e-4 * max(ref, 1e-6), k
        flat = g.flatten()
        idx = torch.linspace(0, flat.numel() - 1, 32).long()
        np.testing.assert_allclose(flat[idx].numpy(), gold["grad_samples"][j], rtol=2e-3, atol=1e-6 + 2e-4 * ref)
    for k in gold.files:
        if k.startswith("gradfull::"):
            name = k.split("::", 1)[1]
            np.testing.assert_allclose(params[name].grad.numpy(), gold[k], rtol=2e-3,
                                       atol=1e-7 + 2e-4 * float(np.abs(gold[k]).max()))


def test_oracle_port_equals_stored_reference_outputs(sd, gold):
    """What test_oracle_port_equals_staged_reference_model compares, without the reference files: the oracle port's
    loss sum, token count and argmax ids on commits 3-5 against the outputs the unmodified reference computed for them
    with the same weights (tests/golden/model_first128.npz: its per-position NLL, already masked by the reference's
    label != 0 mask, and its 'dev' ids), at the live comparison's tolerance."""
    b = golden_batch(3, 6)
    with torch.no_grad():
        loss_sum, n_tok = O.forward(sd, *b, stage="train")
        ids = O.forward(sd, *b, stage="dev")
    ref = float(gold["nll"][3:6].astype(np.float64).sum())
    assert int(n_tok) == int((load_batch_golden()["tar_label"][3:6, 1:] != 0).sum())
    assert np.array_equal(ids.numpy(), gold["dev_ids"][3:6])
    assert abs(ref - loss_sum.item()) <= 1e-5 * abs(ref)


def test_oracle_port_equals_staged_reference_model():
    """oracle/_ref (the unmodified reference files staged by oracle/make_ref.sh, what bench.py's CPU legs time) and
    the oracle port evaluate the same loss and argmax ids on real commits with the same weights."""
    import os
    import subprocess
    import sys
    import torch
    from fira_testlib import ROOT, golden_batch, reference_args
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "Model.py")):
        pytest.skip("oracle/_ref not staged (run `sh oracle/make_ref.sh` where /root/reference exists)")
    code = r"""
import sys, json, torch
sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)
from Model import TransModel
import fira_oracle as O
from fira_testlib import golden_batch, reference_args
torch.manual_seed(0)
m = TransModel(reference_args()); m.eval()
b = golden_batch(3, 6)
with torch.no_grad():
    loss, mask = m(*b, 'train')
    ids = m(*b, 'dev')
    sd = {k: v for k, v in m.state_dict().items()}
    l2, n2 = O.forward(sd, *b, stage='train')
    ids2 = O.forward(sd, *b, stage='dev')
print(json.dumps({'ref': float(loss.sum()), 'port': float(l2), 'n': int(mask.sum()), 'n2': int(n2),
                  'ids_equal': bool(torch.equal(ids, ids2))}))
""" % (ref_dir, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["n"] == out["n2"] and out["ids_equal"]
    assert abs(out["ref"] - out["port"]) <= 1e-5 * abs(out["ref"])
