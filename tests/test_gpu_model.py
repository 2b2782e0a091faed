"""Whole-path parity on the B200: the CUDA TransModel against (a) the committed outputs of the
unmodified reference (tests/golden/model_first128.npz) and (b) the CPU oracle, on real DataSet
commits; fp32 parity mode, tolerance 1e-4 relative (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from fira_testlib import golden_batch, load_model_golden, seeded_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-4


@pytest.fixture(scope="module")
def model():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import copy
    m = copy.deepcopy(seeded_model()).to(DEV)
    m.eval()
    return m


@pytest.fixture(scope="module")
def gold():
    return load_model_golden()


def to_dev(batch):
    return [b.to(DEV) if torch.is_tensor(b) else b for b in batch]


def test_state_dict_is_the_reference_layout(model, gold):
    sd = model.state_dict()
    assert list(sd.keys()) == [str(k) for k in gold["param_keys"]]
    s = np.array([sd[k].double().sum().item() for k in sd])
    np.testing.assert_allclose(s, gold["param_sum"], rtol=0, atol=1e-9)


def test_forward_matches_reference_on_128_commits(model, gold):
    bs = int(gold["batch_size"])
    for bi, lo in enumerate(range(0, 128, bs)):
        batch = to_dev(golden_batch(lo, lo + bs))
        with torch.no_grad():
            loss_sum, n_tok = model(*batch, "train")
            ids = model(*batch, "dev")
        assert int(n_tok) == int(gold["mask_sums"][bi])
        assert abs(loss_sum.item() - gold["loss_sums"][bi]) <= RTOL * gold["loss_sums"][bi]
        assert np.array_equal(ids.cpu().numpy(), gold["dev_ids"][lo:lo + bs]), "argmax ids differ from the reference"


def test_intermediates_match_reference(model, gold):
    from fira_icse_b200 import ops
    batch = to_dev(golden_batch(0, 8))
    sou, tar, attr, mark, ast_change, edge, tar_label, sub_token = batch
    with torch.no_grad():
        code, sub = model.encoder(sou, sou != 0, attr, mark, ast_change, edge, sub_token)
        assert code.shape == (8, 210, 256) and sub.shape == (8, 160, 256)
        memory = torch.cat((code, sub), 1)
        mem_mask = torch.cat((sou != 0, sub_token != 0), 1)
        dec = model.decoder(tar, memory, mem_mask, tar != 0)
        logits = model.out_fc(dec)
        scores, gate = model.copy_net(memory, dec)
        _, nll, _ = ops.HeadFn.apply(False, False, None, memory, dec, mem_mask.to(torch.uint8),
                                     model.shifted_label(tar_label).to(torch.int32).view(-1),
                                     model.out_fc.weight, model.out_fc.bias, *model.copy_net.flat_params())
    real = mem_mask[:4].unsqueeze(-1).cpu().numpy()
    # padding rows are compared too: the dense-row path reproduces them exactly like the reference
    mem = memory[:4, :, ::2].cpu().numpy()                          # the golden keeps every second feature
    np.testing.assert_allclose(mem, gold["full_memory_even"], rtol=RTOL, atol=2e-5)
    np.testing.assert_allclose(mem * real, gold["full_memory_even"] * real, rtol=RTOL, atol=2e-5)
    np.testing.assert_allclose(dec[:4].cpu().numpy(), gold["full_decoder"], rtol=RTOL, atol=2e-5)
    np.testing.assert_allclose(scores[:4].cpu().numpy(), gold["full_copy"], rtol=RTOL, atol=2e-5)
    np.testing.assert_allclose(gate[:4].cpu().numpy(), gold["full_gate"], rtol=RTOL, atol=1e-6)
    np.testing.assert_allclose(logits[:4, :, :256].cpu().numpy(), gold["full_logits_head"], rtol=RTOL, atol=2e-5)
    np.testing.assert_allclose(nll.cpu().numpy(), gold["nll"][:8], rtol=RTOL, atol=1e-5)


def test_packed_edges_equal_dense_edges(model):
    from fira_icse_b200 import PackedEdges
    dense = to_dev(golden_batch(0, 6))
    packed = list(dense)
    packed[5] = PackedEdges.from_coo_lists(golden_batch(0, 6, dense_edge=False)[5], 650, DEV)
    f32 = list(dense)
    f32[5] = dense[5].float()
    with torch.no_grad():
        a = model(*dense, "train")[0].item()
        b = model(*packed, "train")[0].item()
        c = model(*f32, "train")[0].item()
    # split-K partial sums are combined with atomics: equal up to fp32 summation order
    assert abs(a - b) <= 2e-6 * abs(a) and abs(a - c) <= 2e-6 * abs(a)


def test_gradients_match_reference(model, gold):
    n = int(gold["grad_commits"])
    model.zero_grad(set_to_none=True)
    loss_sum, n_tok = model(*to_dev(golden_batch(0, n)), "train")
    loss = loss_sum / n_tok
    loss.backward()
    assert abs(loss.item() - float(gold["grad_loss"])) <= RTOL * float(gold["grad_loss"])
    params = dict(model.named_parameters())
    keys = [str(k) for k in gold["grad_keys"]]
    assert sorted(k for k, p in params.items() if p.grad is not None) == sorted(keys)
    worst = 0.0
    for j, k in enumerate(keys):
        g = params[k].grad
        ref = float(gold["grad_norm"][j])
        if ref < 1e-7:
            # softmax shift-invariance makes d/d(fc_k.bias) and d/d(LinearRes.bias) exactly zero in
            # exact arithmetic: the reference value is round-off noise (~1e-10), only smallness is checked
            assert g.double().norm().item() < 1e-6, k
            continue
        err = abs(g.double().norm().item() - ref) / ref
        worst = max(worst, err)
        assert err <= 5e-4, (k, err)
        flat = g.flatten()
        idx = torch.linspace(0, flat.numel() - 1, 32).long().to(DEV)
        np.testing.assert_allclose(flat[idx].cpu().numpy(), gold["grad_samples"][j], rtol=5e-3,
                                   atol=1e-7 + 5e-4 * ref, err_msg=k)
    for k in gold.files:
        if k.startswith("gradfull::"):
            name = k.split("::", 1)[1]
            np.testing.assert_allclose(params[name].grad.cpu().numpy(), gold[k], rtol=5e-3,
                                       atol=1e-7 + 5e-4 * float(np.abs(gold[k]).max()), err_msg=name)
    print("worst grad-norm rel err", worst)


def test_matches_cpu_oracle_on_other_commits(model):
    import fira_oracle as O
    batch = golden_batch(100, 108)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    with torch.no_grad():
        detail = {}
        ref_sum, ref_tok = O.forward(sd, *batch, stage="train", detail=detail)
        ref_ids = O.forward(sd, *batch, stage="dev")
        loss_sum, n_tok = model(*to_dev(batch), "train")
        ids = model(*to_dev(batch), "dev")
    assert int(n_tok) == int(ref_tok)
    assert abs(loss_sum.item() - ref_sum.item()) <= RTOL * ref_sum.item()
    assert torch.equal(ids.cpu(), ref_ids)


def test_training_steps_reduce_loss_with_dropout(model):
    import copy
    m = copy.deepcopy(model)
    m.train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-4)
    batch = to_dev(golden_batch(32, 48))
    losses = []
    for _ in range(6):
        loss_sum, n_tok = m(*batch, "train")
        loss = loss_sum / n_tok
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)), losses
    assert losses[-1] < losses[0], losses
    # dead blocks never receive gradients (SURVEY.md 2.4)
    assert all(p.grad is None for p in m.dead_parameters())
    assert all(p.grad is not None for p in m.live_parameters())


def test_empty_and_ragged_inputs(model):
    """all-padding message, batch of one, shortest commit"""
    b = to_dev(golden_batch(5, 6))
    b[1] = torch.zeros_like(b[1]); b[6] = torch.zeros_like(b[6])
    with torch.no_grad():
        loss_sum, n_tok = model(*b, "train")
    assert int(n_tok) == 0 and loss_sum.item() == 0.0


# ------------------------------------------------------------------ bf16 throughput mode (tcgen05 GEMMs)
BF16_LOGP_EPS = 5e-2     # bound on |log p_bf16 - log p_fp32| through 12 post-LN layers of bf16 activations


def _head_nll(m, batch):
    """per-position NLL of model `m` (its precision mode) on `batch` through the public sub-modules"""
    from fira_icse_b200 import ops
    sou, tar, attr, mark, ast_change, edge, tar_label, sub_token = batch
    code, sub = m.encoder(sou, sou != 0, attr, mark, ast_change, edge, sub_token)
    memory = torch.cat((code, sub), 1)
    mem_mask = torch.cat((sou != 0, sub_token != 0), 1)
    dec = m.decoder(tar, memory, mem_mask, tar != 0)
    return ops.HeadFn.apply(False, m.precision == "bf16", None, memory, dec, mem_mask.to(torch.uint8),
                            m.shifted_label(tar_label).to(torch.int32).view(-1),
                            m.out_fc.weight, m.out_fc.bias, *m.copy_net.flat_params())


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-30))


def test_bf16_mode_tracks_fp32_mode(model, gold):
    """bf16 activations + tensor-core GEMMs: loss within 2e-2 of the reference, gradients aligned."""
    import copy
    m = copy.deepcopy(model).set_precision("bf16")
    n = int(gold["grad_commits"])
    batch = to_dev(golden_batch(0, n))
    m.zero_grad(set_to_none=True)
    loss_sum, n_tok = m(*batch, "train")
    loss = loss_sum / n_tok
    loss.backward()
    ref = float(gold["grad_loss"])
    assert abs(loss.item() - ref) <= 2e-2 * ref, (loss.item(), ref)
    model.zero_grad(set_to_none=True)
    l32, t32 = model(*batch, "train")
    (l32 / t32).backward()
    p32, p16 = dict(model.named_parameters()), dict(m.named_parameters())
    worst = 1.0
    for k, p in p32.items():
        if p.grad is None:
            assert p16[k].grad is None
            continue
        if p.grad.norm().item() < 1e-6:
            continue
        c = _cos(p.grad, p16[k].grad)
        worst = min(worst, c)
        assert c > 0.98, (k, c)
        r = p16[k].grad.norm().item() / p.grad.norm().item()
        assert 0.9 < r < 1.1, (k, r)
    print("worst bf16-vs-fp32 gradient cosine", worst)
    with torch.no_grad():
        ids16 = m(*batch, "dev")
        ids32 = model(*batch, "dev")
    # argmax ids of the bf16 mode: identical to the fp32 mode wherever the fp32 REFERENCE distribution decides the
    # position by more than the bf16 mode's own log-probability error; every disagreement must be such a near-tie
    # (random-initialised weights: rows are near-uniform over 25,020 entries, top-1/top-2 gaps of 1e-3 are common).
    import fira_oracle as O
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    detail = {}
    with torch.no_grad():
        O.forward(sd, *golden_batch(0, n), stage="train", detail=detail)
    logp = detail["logp"]                                          # fp32 oracle, [n, 30, 25020]
    bad = torch.nonzero(ids16.cpu() != ids32.cpu())
    worst_gap = 0.0
    for i, t in bad.tolist():
        gap = float(logp[i, t, int(ids32[i, t])] - logp[i, t, int(ids16[i, t])])
        worst_gap = max(worst_gap, abs(gap))
        assert abs(gap) <= BF16_LOGP_EPS, f"commit {i} position {t}: bf16 argmax differs beyond a near-tie ({gap:.3e})"
    print(f"bf16 argmax: {len(bad)} of {ids32.numel()} positions differ, all near-ties (worst fp32 gap {worst_gap:.2e})")
    # and the per-position NLL of the bf16 mode stays within the same bound of the fp32 reference
    from fira_icse_b200 import ops
    with torch.no_grad():
        nll32 = detail["nll"]
        _, nll16, _ = _head_nll(m, batch)
    keep = nll32 != 0
    assert (nll16.cpu()[keep] - nll32[keep]).abs().max().item() <= BF16_LOGP_EPS


def test_bf16_training_reduces_loss(model):
    import copy
    m = copy.deepcopy(model).set_precision("bf16")
    m.train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-4)
    batch = to_dev(golden_batch(32, 48))
    losses = []
    for _ in range(6):
        loss_sum, n_tok = m(*batch, "train")
        loss = loss_sum / n_tok
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses


def test_trimmed_batch_equals_padded_batch(model):
    """loader-side padding trimming (data.trim_batch_host): same loss, same gradients, fewer rows"""
    from fira_icse_b200 import PackedEdges
    from fira_icse_b200.data import trim_batch_host
    n = 12
    b = golden_batch(0, n, dense_edge=False)
    rowptr, col, val = PackedEdges.pack_host(b[5], 650)
    full = [b[0], b[1], None, b[3], b[4], (rowptr, col, val), b[6], b[7]]
    trim = trim_batch_host(full, model.vocab_size)
    assert trim[0].shape[1] < 210 and trim[4].shape[1] < 280

    def run(lst):
        n_nodes = lst[0].shape[1] + lst[7].shape[1] + lst[4].shape[1]
        dev_lst = [x.to(DEV) if torch.is_tensor(x) else x for x in lst]
        dev_lst[5] = PackedEdges.from_host(*lst[5], n, n_nodes, DEV)
        model.zero_grad(set_to_none=True)
        ls, nt = model(*dev_lst, "train")
        (ls / nt).backward()
        with torch.no_grad():
            ids = model(*dev_lst, "dev")
        return ls.item(), int(nt), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}, ids
    l_full, n_full, g_full, ids_full = run(full)
    l_trim, n_trim, g_trim, ids_trim = run(trim)
    assert n_full == n_trim and abs(l_full - l_trim) <= 2e-6 * abs(l_full)
    for k in g_full:
        scale = g_full[k].abs().max().item()
        if scale < 1e-6:          # shift-invariant biases: exactly zero in exact arithmetic, round-off noise here
            continue
        assert (g_full[k] - g_trim[k]).abs().max().item() <= 1e-4 * scale + 1e-9, k
    # argmax ids: vocabulary and code-copy ids identical, sub-token copy ids shifted by the trimmed code padding
    V, c0 = model.vocab_size, trim[0].shape[1]
    expect = torch.where(ids_full >= V + 210, ids_full - (210 - c0), ids_full)
    assert torch.equal(ids_trim, expect)
