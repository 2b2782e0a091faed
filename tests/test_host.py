"""CPU-side checks: C-ABI library loads and exports every declared symbol, module surface /
state_dict layout, packed-edge collation, synthetic generator, loud failure without a GPU."""
import ctypes
import os

import numpy as np
import pytest
import torch

from fira_testlib import ROOT, golden_batch, load_batch_golden, load_model_golden, reference_args, seeded_model


def test_library_exports_every_symbol_the_header_declares():
    import __graft_entry__ as g
    g.build()
    from fira_icse_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos) >= 25
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in protos:
        assert hasattr(handle, name), f"{name} declared in include/fira_b200.h but not exported"
    lib = _lib.lib()
    assert lib.fira_version() >= 2 and lib.fira_built_arch() == 100
    out = os.popen(f"nm -D --defined-only {_lib.LIB_PATH}").read()
    exported = {l.split()[-1] for l in out.splitlines() if " T fira_" in l}
    assert exported == set(protos), exported ^ set(protos)     # nothing exported that the header hides


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """the boundary is a C ABI: include/fira_b200.h must compile as C99 and a C program must link against the
    library and call it (version / error string / a host entry point; no GPU work)"""
    import shutil
    import subprocess
    from fira_icse_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "abi.c"
    src.write_text(r'''
#include <stdio.h>
#include "fira_b200.h"
int main(void) {
  int pairs[2] = {0, 0};                 /* AST node 0 - code token 0 */
  int deg[8], col[32], nnz = -1;
  double val[32];
  int rc = fira_host_build_adjacency(0, 0, 0, 0, pairs, 1, 0, 0, 0, 0, 1, 1, 4, 2, 2, deg, col, val, 32, &nnz);
  if (rc != 0) { printf("error %d: %s\n", rc, fira_last_error_string()); return 1; }
  rc = fira_host_build_adjacency(0, 0, 0, 0, pairs, 1, 0, 0, 0, 0, 1, 1, 4, 2, 2, deg, col, val, 2, &nnz);
  printf("%d %d %d %d %s\n", fira_version(), fira_built_arch(), nnz, rc, rc ? "capacity-error-reported" : "");
  return 0;
}
''')
    exe = tmp_path / "abi"
    lib_dir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe), "-L", lib_dir, "-l:libfira_b200.so", f"-Wl,-rpath,{lib_dir}"])
    out = subprocess.check_output([str(exe)], text=True).split()
    assert out[:3] == [str(_lib.lib().fira_version()), "100", "14"] and int(out[3]) != 0 and out[4] == "capacity-error-reported", out


def test_sass_is_sm100():
    from fira_icse_b200 import _lib
    out = os.popen(f"/usr/local/cuda/bin/cuobjdump -lelf {_lib.LIB_PATH} 2>/dev/null").read()
    assert "sm_100a" in out, out


def test_state_dict_layout_and_seeded_init_match_the_reference():
    gold = load_model_golden()
    sd = seeded_model().state_dict()
    assert len(sd) == 338
    assert list(sd.keys()) == [str(k) for k in gold["param_keys"]]
    assert [sd[k].numel() for k in sd] == list(gold["param_numel"])
    # the float64 sums are split across CPU threads, so their last bits depend on how many threads take part: sum on
    # the 8 threads tests/golden/make_golden.py summed with
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        s = np.array([sd[k].double().sum().item() for k in sd])
        a = np.array([sd[k].double().abs().sum().item() for k in sd])
    finally:
        torch.set_num_threads(threads)
    assert np.array_equal(s, gold["param_sum"]) and np.array_equal(a, gold["param_abs"])   # bit-identical init


def test_dead_parameters_are_the_74_gradless_tensors():
    m = seeded_model()
    gold = load_model_golden()
    live = {id(p) for p in m.live_parameters()}
    names = sorted(k for k, p in m.named_parameters() if id(p) in live)
    assert names == sorted(str(k) for k in gold["grad_keys"])
    assert len(m.dead_parameters()) == 74


def test_position_encoding_equals_oracle_table():
    import fira_oracle as O
    from fira_icse_b200 import position_encoding
    for n in (30, 210):
        assert torch.allclose(position_encoding(n, 256), O.position_table(n, 256), atol=1e-7, rtol=0)


def test_no_cpu_fallback():
    from fira_icse_b200 import FiraLibraryError
    m = seeded_model()
    b = golden_batch(0, 2)
    with pytest.raises((FiraLibraryError, RuntimeError)):
        m(*b, "train")
    with pytest.raises((FiraLibraryError, RuntimeError)):
        m.out_fc(torch.zeros(2, 256))


def test_pack_host_reproduces_reference_dense_adjacency():
    from fira_icse_b200 import PackedEdges
    coo = golden_batch(0, 5, dense_edge=False)[5]
    dense = golden_batch(0, 5)[5]
    rowptr, col, val = PackedEdges.pack_host(coo, 650)
    pe = PackedEdges(rowptr, col, val, 5, 650, True)
    assert torch.equal(pe.to_dense(torch.float32), dense.float())
    assert rowptr.dtype == torch.int32 and col.dtype == torch.int32 and val.dtype == torch.float32
    # Dataset.py adjacency is symmetric: to 1 ulp in float64, exactly after the model's .float() cast
    assert torch.equal(dense.float(), dense.float().transpose(1, 2))
    # duplicates are summed like scipy's toarray()
    r, c, v = coo[0]
    rp2, c2, v2 = PackedEdges.pack_host([(np.concatenate((r, r[:3])), np.concatenate((c, c[:3])),
                                          np.concatenate((v, v[:3])))], 650)
    d2 = PackedEdges(rp2, c2, v2, 1, 650, True).to_dense()
    exp = dense[:1].clone()
    for k in range(3):
        exp[0, r[k], c[k]] += v[k]
    assert torch.allclose(d2, exp.float().double(), atol=1e-7)


def test_synthetic_generator_follows_the_dataset_distribution():
    from fira_icse_b200.synth import N_NODES, synth_batch, synth_stress_graphs
    ids, coo = synth_batch(0, 256)
    n_code = (ids["sou"] != 0).sum(1)
    n_sub = (ids["sub_token"] != 0).sum(1)
    n_ast = (ids["ast_change"] != 0).sum(1)
    n_tok = (ids["tar_label"][:, 1:] != 0).sum(1)
    offdiag = np.array([len(r) - N_NODES for r, _, _ in coo])
    assert 85 < n_code.mean() < 115 and n_code.max() <= 200
    assert 20 < n_sub.mean() < 34 and n_sub.max() <= 102
    assert 24 < n_ast.mean() < 40 and n_ast.max() <= 157
    assert 6 < n_tok.mean() < 10
    assert 330 < offdiag.mean() < 470, offdiag.mean()          # DataSet: mean 401 directed off-diagonal entries
    ids2, _ = synth_batch(0, 4)
    assert all(np.array_equal(ids[k][:4], ids2[k]) for k in ids)   # seeded per commit index
    r, c, v = coo[0]
    a = np.zeros((N_NODES, N_NODES)); a[r, c] = v
    assert np.allclose(a, a.T) and np.allclose(np.diag(a)[400:], 1.0)
    lab = ids["tar_label"]
    assert lab.max() < 24650 + 370 and ((lab >= 24650).sum() > 0)
    g = synth_stress_graphs(0, 1, n_nodes=256, edges_per_relation=512)
    assert g[0][0].max() < 256


def test_shard_range_covers_everything_once():
    from fira_icse_b200.parallel import shard_range
    for n in (0, 1, 7, 7661):
        for w in (1, 2, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))


def test_flat_adam_has_no_cpu_path():
    """optim.FlatAdam re-homes CUDA parameters only: CPU parameters raise instead of falling back"""
    import torch
    from fira_icse_b200 import FiraLibraryError
    from fira_icse_b200.optim import FlatAdam, cat_rows, grad_dest, mirror_of
    p = torch.nn.Parameter(torch.zeros(8, 8))
    with pytest.raises(FiraLibraryError):
        FlatAdam([p], lr=1e-3)
    # the lookups used by the backward passes treat ordinary tensors as "not re-homed"
    assert mirror_of(p) is None and grad_dest((p,), (8, 8)) is None
    assert torch.equal(cat_rows((p.data, p.data)), torch.cat((p.data, p.data), 0))


def test_flat_layout_keeps_fused_operands_adjacent():
    """optim.plan_layout on the real parameter set: every group of TransModel.flat_groups() lies back to back (the q|k,
    q|k|v and 12-way k|v weights / biases and every LayerNorm (weight, bias) pair are single views for ops.py), every
    tensor starts on a 64-element boundary unless it continues a group, nothing overlaps, and the live parameters are
    exactly the ones that receive gradients (264 of the 338)."""
    from fira_testlib import seeded_model
    from fira_icse_b200.optim import ALIGN, plan_layout
    m = seeded_model()
    params = [p for p in m.live_parameters() if p.requires_grad]
    groups = m.flat_groups()
    offs, n = plan_layout(params, groups)
    off = {id(p): o for p, o in zip(params, offs)}
    assert len(params) == 264 and n % ALIGN == 0
    spans = sorted((o, o + p.numel()) for p, o in zip(params, offs))
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:])) and spans[-1][1] <= n
    in_group = set()
    for g in groups:
        assert off[id(g[0])] % ALIGN == 0
        for a, b in zip(g, g[1:]):
            assert off[id(b)] == off[id(a)] + a.numel()
            in_group.add(id(b))
    assert all(off[id(p)] % ALIGN == 0 for p in params if id(p) not in in_group)
    # the groups ops.py relies on
    dec, enc = m.decoder, m.encoder
    kv = [t for c in dec.cross_attention_list for t in (c.fc_k.weight, c.fc_v.weight)]
    assert off[id(kv[-1])] - off[id(kv[0])] == 11 * 256 * 256
    a0 = dec.attention_list[0]
    assert off[id(a0.fc_v.weight)] == off[id(a0.fc_q.weight)] + 2 * 256 * 256
    c0 = enc.combination_list2[0].linear_layers
    assert off[id(c0[1].bias)] == off[id(c0[0].bias)] + 256
    # two optimizers (head/decoder | encoder): groups split cleanly, none straddles the cut
    dec_ids = {id(p) for p in list(m.decoder.parameters()) + list(m.out_fc.parameters()) + list(m.copy_net.parameters())}
    pa = [p for p in params if id(p) in dec_ids]
    pb = [p for p in params if id(p) not in dec_ids]
    for part in (pa, pb):
        o2, _ = plan_layout(part, groups)
        o2 = {id(p): o for p, o in zip(part, o2)}
        for g in groups:
            if all(id(p) in o2 for p in g):
                for a, b in zip(g, g[1:]):
                    assert o2[id(b)] == o2[id(a)] + a.numel()
            else:
                assert not any(id(p) in o2 for p in g)


def test_timeline_summary_splits_replays_evenly():
    """tools/timeline_summary.py: a trace of n identical graph replays is cut by kernel count even when a gap inside a
    step is longer than the gaps between steps (the case that broke the gap heuristic)"""
    import io
    import sys as _sys
    _sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import timeline_summary as TS
    ev, t = [], 0.0
    for step in range(3):
        for i, name in enumerate(["void a_kernel<int>(int)", "void b_kernel(float*)", "void a_kernel<int>(int)", "c_kernel()"]):
            gap = 500.0 if i == 2 else 1.0                     # a long stall INSIDE every step
            t += gap
            ev.append({"name": name, "ts": t, "dur": 5.0, "cat": "kernel", "args": {"stream": 7 + (i % 2)}})
            t += 5.0
        t += 20.0                                              # the gap between steps is shorter than the stall
    steps = TS.split_steps(ev, 3)
    assert [len(s) for s in steps] == [4, 4, 4]
    out = io.StringIO()
    TS.summarize(steps[1], out=out)
    text = out.getvalue()
    assert "kernels 4" in text and "a_kernel<int>" in text
