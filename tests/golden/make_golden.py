#!/usr/bin/env python
"""Generate the committed golden fixtures from the UNMODIFIED reference.

Runs only in the build container (needs /root/reference). Nothing under tests/,
bench.py or smoke() reads /root/reference at run time: they read the files this
script wrote into tests/golden/.

What it does
  1. slices the first N_COMMITS commits out of the reference DataSet/*.json,
  2. runs the reference's own Dataset.TransDataset.process_data on that slice
     (monkey-patching only the split sizes, Dataset.py:10-12) and un-shuffles it,
  3. builds the reference Model.TransModel under torch.manual_seed(0) with the real
     vocabulary sizes (run_model.py:27-56) and records, in eval mode:
       per-position NLL, loss/mask sums, 'dev' argmax ids, encoder memory, decoder
       output, copy scores, gate, vocab-logit slices, and the gradients of
       loss_sum/mask_sum for the first GRAD_COMMITS commits,
  4. writes   tests/golden/raw_first128.json.gz   (raw inputs + vocabularies)
              tests/golden/batch_first128.npz     (reference-built id arrays + COO edges)
              tests/golden/model_first128.npz     (reference model outputs)

Usage:  python tests/golden/make_golden.py
"""
import gzip
import json
import os
import pickle
import sys
import tempfile

import numpy as np
import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
N_COMMITS = 128
GRAD_COMMITS = 16
FULL_COMMITS = 4   # commits whose intermediate tensors are stored in full
RAW_NAMES = ["difftoken", "diffatt", "diffmark", "msg", "variable", "change", "ast",
             "edge_change_code", "edge_change_ast", "edge_ast_code", "edge_ast"]


class DotDict(dict):
    def __getattr__(self, k):
        return self[k]


def main():
    torch.set_num_threads(8)
    scratch = tempfile.mkdtemp(prefix="fira_golden_")
    os.symlink(os.path.join(REF, "DataSet"), os.path.join(scratch, "DataSet"))
    os.symlink(os.path.join(REF, "VOCAB_UPPER_CASE"), os.path.join(scratch, "VOCAB_UPPER_CASE"))
    os.chdir(scratch)
    sys.path.insert(0, REF)

    # ---------------------------------------------------------------- raw slice
    raw = {}
    for n in RAW_NAMES:
        raw[n] = json.load(open(os.path.join(REF, "DataSet", n + ".json")))[:N_COMMITS]
    word_vocab = json.load(open(os.path.join(REF, "DataSet", "word_vocab.json")))
    ast_vocab = json.load(open(os.path.join(REF, "DataSet", "ast_change_vocab.json")))
    upper = json.load(open(os.path.join(REF, "VOCAB_UPPER_CASE")))
    with gzip.open(os.path.join(HERE, "raw_first128.json.gz"), "wt") as f:
        json.dump({"raw": raw, "word_vocab": word_vocab, "ast_change_vocab": ast_vocab,
                   "VOCAB_UPPER_CASE": upper}, f)

    # ------------------------------------------------- reference graph builder
    import Dataset as RefDataset
    RefDataset.num_train, RefDataset.num_valid, RefDataset.num_test = N_COMMITS, 0, 0
    args = DotDict(sou_len=210, tar_len=30, att_len=25, ast_change_len=280, sub_token_len=160,
                   lr=1e-4, dropout_rate=0.1, num_head=8, embedding_dim=256,
                   vocab_size=len(word_vocab), ast_change_vocab_size=len(ast_vocab))
    ds = object.__new__(RefDataset.TransDataset)
    ds.data_name = "train"
    ds.diff_len, ds.msg_len, ds.att_len = 210, 30, 25
    ds.ast_change_len, ds.sub_token_len = 280, 160
    ds.graph_len = 650
    ds.vocab, ds.ast_change_vocab = word_vocab, ast_vocab
    raw_copy = json.loads(json.dumps(raw))  # process_data mutates its inputs
    ds.process_data(raw_copy["difftoken"], raw_copy["diffatt"], raw_copy["diffmark"], raw_copy["msg"],
                    raw_copy["variable"], raw_copy["change"], raw_copy["ast"],
                    raw_copy["edge_change_code"], raw_copy["edge_change_ast"],
                    raw_copy["edge_ast_code"], raw_copy["edge_ast"])
    data = pickle.load(open("processed_train.pkl", "rb"))
    order = json.load(open("all_index"))["train"]
    inv = np.argsort(np.array(order))           # position in shuffled list of commit i
    arrs = [np.asarray(data[i])[inv] if i != 5 else [data[5][j] for j in inv] for i in range(8)]
    sou, tar, attr, mark, ast_change, edges, tar_label, sub_token = arrs
    ptr = [0]
    rows, cols, vals = [], [], []
    for e in edges:
        e = e.tocoo()
        rows.append(e.row.astype(np.int16)); cols.append(e.col.astype(np.int16))
        vals.append(e.data.astype(np.float64)); ptr.append(ptr[-1] + e.nnz)
    np.savez_compressed(
        os.path.join(HERE, "batch_first128.npz"),
        sou=sou.astype(np.int16), tar=tar.astype(np.int16), attr=attr.astype(np.int16),
        mark=mark.astype(np.int8), ast_change=ast_change.astype(np.int16),
        tar_label=tar_label.astype(np.int16), sub_token=sub_token.astype(np.int16),
        edge_ptr=np.array(ptr, np.int32), edge_row=np.concatenate(rows),
        edge_col=np.concatenate(cols), edge_val=np.concatenate(vals))

    # ------------------------------------------------------- reference model
    import Model as RefModel
    import torch.nn.functional as F
    torch.manual_seed(0)
    model = RefModel.TransModel(args)
    model.eval()
    sd = model.state_dict()
    keys = list(sd.keys())
    out = {"param_keys": np.array(keys),
           "param_sum": np.array([sd[k].double().sum().item() for k in keys]),
           "param_abs": np.array([sd[k].double().abs().sum().item() for k in keys]),
           "param_numel": np.array([sd[k].numel() for k in keys])}

    def batch(lo, hi):
        dense = np.stack([edges[i].toarray() for i in range(lo, hi)])
        return [torch.from_numpy(np.ascontiguousarray(a[lo:hi])).long() if a is not None else None
                for a in (sou, tar, attr, mark, ast_change)] + \
               [torch.from_numpy(dense)] + \
               [torch.from_numpy(np.ascontiguousarray(a[lo:hi])).long() for a in (tar_label, sub_token)]

    nll_all, ids_all, loss_sums, mask_sums = [], [], [], []
    mem_abs, dec_abs = [], []
    BS = 32
    with torch.no_grad():
        for lo in range(0, N_COMMITS, BS):
            b = batch(lo, lo + BS)
            ls, ms = model(*b, "train")
            ids = model(*b, "dev")
            loss_sums.append(ls.item()); mask_sums.append(ms.item()); ids_all.append(ids.numpy())
            # re-run the pieces the way run_model.py:204-265 does, to record intermediates
            sou_mask = b[0] != 0
            sub_mask = b[7] != 0
            code_em, sub_em = model.encoder(b[0], sou_mask, b[2], b[3], b[4], b[5], b[7])
            memory = torch.cat((code_em, sub_em), 1)
            mem_mask = torch.cat((sou_mask, sub_mask), 1)
            dec = model.decoder(b[1], memory, mem_mask, b[1] != 0)
            logits = model.out_fc(dec)
            gen = F.softmax(logits, -1)
            copy, gate = model.copy_net(memory, dec)
            copy_m = torch.masked_fill(copy, mem_mask.unsqueeze(1) == 0, -1e9)
            copy_p = F.softmax(copy_m, -1)
            full = torch.cat((gate[:, :, 0:1] * gen, gate[:, :, 1:2] * copy_p), -1)
            logp = torch.log(full.clamp(min=1e-10, max=1))
            label = torch.cat([b[6], torch.zeros(b[6].size(0), 1, dtype=torch.long)], -1)[:, 1:]
            nll = -logp.gather(-1, label.unsqueeze(-1)).squeeze(-1) * (label != 0)
            nll_all.append(nll.numpy())
            mem_abs.append((memory.abs() * mem_mask.unsqueeze(-1)).sum((1, 2)).numpy())
            dec_abs.append(dec.abs().sum((1, 2)).numpy())
            if lo == 0:
                n = FULL_COMMITS
                # every second feature of the encoder memory: the whole of it would push the file past 1 MB
                out.update(full_memory_even=memory[:n, :, ::2].numpy(), full_decoder=dec[:n].numpy(),
                           full_copy=copy[:n].numpy(), full_gate=gate[:n].numpy(),
                           full_logits_head=logits[:n, :, :256].numpy(),
                           full_logp_max=logp[:n].max(-1).values.numpy())
    out.update(nll=np.concatenate(nll_all), dev_ids=np.concatenate(ids_all),
               loss_sums=np.array(loss_sums), mask_sums=np.array(mask_sums),
               mem_abs=np.concatenate(mem_abs), dec_abs=np.concatenate(dec_abs), batch_size=BS)

    # gradients (eval mode == dropout off; identical to train mode with p=0)
    b = batch(0, GRAD_COMMITS)
    model.zero_grad()
    ls, ms = model(*b, "train")
    (ls / ms).backward()
    g_keys, g_norm, g_sum, g_head = [], [], [], []
    for k, p in model.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.double()
        g_keys.append(k); g_norm.append(g.norm().item()); g_sum.append(g.sum().item())
        flat = p.grad.flatten()
        idx = torch.linspace(0, flat.numel() - 1, 32).long()
        g_head.append(flat[idx].numpy())
    out.update(grad_keys=np.array(g_keys), grad_norm=np.array(g_norm), grad_sum=np.array(g_sum),
               grad_samples=np.stack(g_head), grad_loss=float((ls / ms).item()),
               grad_commits=GRAD_COMMITS)
    # small parameters: keep the whole gradient (they see every code path)
    for k in ["copy_net.LinearRes.weight", "copy_net.LinearProb.weight", "copy_net.LinearProb.bias",
              "encoder.gcn_list.0.fc1.bias", "encoder.gcn_list.5.layernorm.weight",
              "encoder.mark_embedding.weight", "decoder.cross_attention_list.0.fc_k.bias",
              "encoder.combination_list2.0.linear_layers.2.bias"]:
        out["gradfull::" + k] = dict(model.named_parameters())[k].grad.numpy()
    np.savez_compressed(os.path.join(HERE, "model_first128.npz"), **out)
    print("wrote goldens;", {k: (v.shape if hasattr(v, 'shape') else v) for k, v in out.items()
                              if not k.startswith('param_')})
    print("loss_sums", loss_sums, "mask_sums", mask_sums)


if __name__ == "__main__":
    main()
