"""Generates the committed golden vectors under tests/golden/.

Runs in the BUILD container only (needs /root/reference).  Three fixtures:

  pool_golden.npz     inputs + outputs of the reference's OWN code, imported from
                      /root/reference/retriever/encoders.py: average_pool (:56-58) followed by
                      F.normalize (:76) for the E5 tail, hidden[:, 0] + F.normalize (:115-117) for
                      the BGE tail, and a tiny-config E5Encoder.forward / BGEEncoder.forward run
                      end to end (last_hidden_state captured with a forward hook).
  aligner_golden.npz  inputs + outputs of the reference's aligner scoring expression
                      (knowledge_graph/models.py:1532-1538): torch.matmul + torch.topk on CPU.
  search_golden.npz, search_golden_1024.npz
                      seeded flat-IP search cases answered by the ORACLE (fp64 accumulate).  The
                      reference's FAISS cannot run here, so this fixture pins the oracle against
                      regressions, not against FAISS ("parity unpinned", see oracle/flat_ip_oracle.c).

Usage:  python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")


def make_pool():
    from retriever.encoders import BGEEncoder, E5Encoder, average_pool  # the reference's own code
    import torch.nn.functional as F
    from transformers import BertConfig

    g = torch.Generator().manual_seed(777)
    out = {}
    # case A: ragged right-padded masks, H=1024
    B, S, H = 6, 37, 1024
    h = torch.randn(B, S, H, generator=g)
    lens = torch.tensor([37, 1, 5, 20, 36, 12])
    m = (torch.arange(S)[None, :] < lens[:, None]).to(torch.int64)
    out["a_hidden"], out["a_mask"] = h.numpy(), m.numpy()
    out["a_avg"] = average_pool(h, m).numpy()
    out["a_e5"] = F.normalize(average_pool(h, m), p=2, dim=1).numpy()
    out["a_bge"] = F.normalize(h[:, 0], p=2, dim=1).numpy()
    # case B: odd sizes (H not a multiple of 4, S not a multiple of 32), holes in the mask
    B, S, H = 3, 9, 50
    h = torch.randn(B, S, H, generator=g)
    m = torch.tensor([[1, 0, 1, 1, 0, 0, 1, 0, 1], [1] * 9, [0, 0, 0, 0, 1, 0, 0, 0, 0]], dtype=torch.int64)
    out["b_hidden"], out["b_mask"] = h.numpy(), m.numpy()
    out["b_avg"] = average_pool(h, m).numpy()
    out["b_e5"] = F.normalize(average_pool(h, m), p=2, dim=1).numpy()
    # case C: bf16 hidden states (trainer autocast), all-ones mask
    B, S, H = 4, 16, 256
    h = torch.randn(B, S, H, generator=g).to(torch.bfloat16)
    m = torch.ones(B, S, dtype=torch.int64)
    out["c_hidden_f32"] = h.float().numpy()  # exactly representable bf16 values
    out["c_mask"] = m.numpy()
    out["c_e5_bf16ref"] = F.normalize(average_pool(h, m), p=2, dim=1).float().numpy()
    out["c_e5_f32ref"] = F.normalize(average_pool(h.float(), m), p=2, dim=1).numpy()
    # case D: the encoders end to end on a tiny BertConfig
    cfg = BertConfig(vocab_size=97, hidden_size=64, num_hidden_layers=2, num_attention_heads=4,
                     intermediate_size=128, max_position_embeddings=32)
    torch.manual_seed(5)
    ids = torch.randint(0, 97, (5, 11))
    lens = torch.tensor([11, 3, 7, 1, 9])
    mask = (torch.arange(11)[None, :] < lens[:, None]).to(torch.int64)
    for name, cls in (("e5", E5Encoder), ("bge", BGEEncoder)):
        torch.manual_seed(11)
        enc = cls(cfg).eval()
        with torch.no_grad():
            emb = enc(ids, mask)
            hidden = super(cls, enc).forward(input_ids=ids, attention_mask=mask, return_dict=True).last_hidden_state
        out[f"d_{name}_hidden"] = hidden.numpy()
        out[f"d_{name}_out"] = emb.numpy()
    out["d_mask"] = mask.numpy()
    np.savez_compressed(os.path.join(HERE, "pool_golden.npz"), **out)


def make_aligner():
    g = torch.Generator().manual_seed(4242)
    out = {}
    for name, (C, T, d, k) in {"s": (2, 37, 64, 20), "m": (3, 300, 128, 20), "few": (2, 7, 64, 20)}.items():
        q = torch.nn.functional.normalize(torch.randn(C, d, generator=g), dim=1)
        t = torch.nn.functional.normalize(torch.randn(T, d, generator=g), dim=1)
        # verbatim knowledge_graph/models.py:1532-1538
        sims = torch.matmul(q, t.T)
        scores, indices = torch.topk(sims, k=min(k, T), dim=1)
        out[f"{name}_q"], out[f"{name}_t"] = q.numpy(), t.numpy()
        out[f"{name}_scores"], out[f"{name}_indices"] = scores.numpy(), indices.numpy()
        out[f"{name}_k"] = np.int64(k)
    np.savez_compressed(os.path.join(HERE, "aligner_golden.npz"), **out)


def make_search():
    from oracle import oracle

    out = {}
    rng = np.random.default_rng(20261018)
    cases = {"unit_64": (2000, 64, 7, 10), "unit_1024": (256, 1024, 5, 20), "kgtn": (6, 64, 2, 10)}
    for name, (n, d, nq, k) in cases.items():
        xb = rng.standard_normal((n, d)).astype(np.float32)
        xb /= np.linalg.norm(xb, axis=1, keepdims=True)
        xq = rng.standard_normal((nq, d)).astype(np.float32)
        xq /= np.linalg.norm(xq, axis=1, keepdims=True)
        D, I = oracle.flat_ip_search(xb, xq, k, accum="f64")
        out[f"{name}_seed_note"] = np.array("default_rng(20261018), cases in dict order")
        out[f"{name}_xb"], out[f"{name}_xq"], out[f"{name}_D"], out[f"{name}_I"] = xb, xq, D, I
        out[f"{name}_k"] = np.int64(k)
    # integer-valued case with many exact ties (answer is precision-independent)
    xb = rng.integers(-2, 3, size=(500, 64)).astype(np.float32)
    xb[100:110] = xb[5]  # duplicates -> exact ties, lower id must win
    xq = rng.integers(-2, 3, size=(4, 64)).astype(np.float32)
    D, I = oracle.flat_ip_search(xb, xq, 16, accum="f64")
    out["ties_xb"], out["ties_xq"], out["ties_D"], out["ties_I"], out["ties_k"] = xb, xq, D, I, np.int64(16)
    # two files, each under 1 MB: the 256 x 1024 case on its own (tests/helpers.py:load_search_golden reads both)
    big = {f: out.pop(f) for f in list(out) if f.startswith("unit_1024_")}
    np.savez_compressed(os.path.join(HERE, "search_golden.npz"), **out)
    np.savez_compressed(os.path.join(HERE, "search_golden_1024.npz"), **big)


if __name__ == "__main__":
    make_pool()
    make_aligner()
    make_search()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
