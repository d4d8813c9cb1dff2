"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference operators.

The reference ships no golden vectors or seeds for this path (SURVEY.md 8(c): its tests are
property-style on unseeded random data), so these fixtures are produced by executing the reference's
own compiled operators (`oracle/_ref`, built by oracle/build_ref.py from the reference checkout that
MAGICPIG_REFERENCE names) on seeded inputs.  The fixtures are committed, so the tests that read them
need neither the reference nor its binaries.

    python tests/golden/make_golden.py          # rewrites tests/golden/*.npz and reference_api.json

Files
  small_chain.npz  B=2 Hq=4 Hkv=2 d=128 K=6 L=24 n=128 M=160: all inputs stored + reference outputs
                   of LSH.fill/batch_retrieve/get_mask and SparseAttentionServer.attention_wrapper,
                   plus one all-miss query row set (nnz = 0 edge).
  c1_chain.npz     BASELINE config[0]: 1 head, seq 4096, d 128, K 10, L 150 (M = 4224); inputs are
                   regenerated from seeds by magicpig_b200.synth (checksums stored), outputs stored.
  operator_cases.npz  LSH.fill/batch_retrieve/get_mask on library/lsh/test.py's case shapes and
                   SparseAttentionServer.attention_wrapper on random index sets (tests/test_oracle_cpu.py
                   *_vs_live_reference): inputs regenerated from seeded torch generators (checksums
                   stored), the reference's outputs stored.
  reference_api.json  the reference's call surface read from its sources (never imported): the
                   LSHSparseAttnServer methods with parameter names and literal defaults, the
                   models/llama.py and models/attnserver.py call sites (positional count + keyword
                   names), the pybind `.def` lists and the C++ member parameter names -- what
                   tests/test_signature_compat.py binds this repo's mirrors against.
"""
from __future__ import annotations

import ast
import hashlib
import json
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from magicpig_b200 import synth  # noqa: E402
from oracle import ref_loader  # noqa: E402

# library/lsh/test.py's case shapes: (K, L, seq, delta, group, bsz)
PROBE_CASES = [(4, 50, 1024, 128, 4, 1), (8, 100, 1024, 128, 8, 2), (8, 50, 4096, 1024, 4, 1)]


def u16(t: torch.Tensor) -> np.ndarray:
    return t.contiguous().view(torch.int16).numpy().view(np.uint16)


def checksum(*tensors) -> str:
    h = hashlib.sha256()
    for t in tensors:
        t = t.contiguous()
        if t.dtype == torch.bfloat16:
            t = t.view(torch.int16)
        h.update(t.numpy().tobytes())
    return h.hexdigest()


def run_reference_chain(B, Hq, Hkv, d, K, L, n, M, key, value, key_norm, hash_func, query, qcodes=None):
    """key/value (B,Hkv,n,d) bf16, key_norm (B,Hkv,n), query (B,Hq,1,d) bf16 -> dict of reference outputs."""
    lsh_m, sa_m, flavour = ref_loader.load()
    kcodes = synth.hash_keys(key, hash_func, K, L)  # (B,Hkv,L,n) int16
    if qcodes is None:
        qcodes = synth.hash_queries_ref(query, hash_func, K, L)
    sc, si = kcodes.sort()
    R = lsh_m.LSH()
    R.alloc(K, L, 1, Hq, Hkv, B, M)
    for b in range(B):
        R.fill(0, b, sc[b].contiguous(), si[b].int().contiguous())
    results = torch.zeros((B * Hq, M), dtype=torch.int32)
    nnz = torch.zeros((B * Hq,), dtype=torch.int32)
    R.batch_retrieve(0, qcodes.contiguous(), results, nnz)
    mask = R.get_mask().clone().view(torch.uint8).reshape(B * Hq, M)
    S = sa_m.SparseAttentionServer()
    S.alloc(1, Hq, Hkv, d, B, M)
    for b in range(B):
        S.fill(0, b, key[b].contiguous(), value[b].contiguous(), key_norm[b].contiguous())
    out = torch.zeros((B * Hq, d), dtype=torch.bfloat16)
    mve = torch.zeros((2, B * Hq), dtype=torch.float32)
    q2 = query.reshape(B * Hq, d).contiguous()
    qn = q2.float().norm(p=2, dim=-1)
    S.attention_wrapper(0, K, L, out, mve, q2, qn, results, nnz)
    # results as sorted sets, flattened with offsets (order is unspecified by the reference)
    flat, offs = [], [0]
    for h in range(B * Hq):
        s = results[h, : nnz[h]].sort().values
        flat.append(s)
        offs.append(offs[-1] + int(nnz[h]))
    return dict(kcodes=kcodes.numpy(), qcodes=qcodes.numpy(), nnz=nnz.numpy(),
                results_sorted=torch.cat(flat).numpy() if flat else np.zeros(0, np.int32),
                results_offsets=np.array(offs, np.int64), mask=mask.numpy(), out_bf16=u16(out), mve=mve.numpy(),
                flavour=np.array(flavour))


def make_small():
    B, Hq, Hkv, d, K, L, n, M = 2, 4, 2, 128, 6, 24, 128, 160
    hf = synth.make_hash_func(d, K, L, seed=10)
    q = synth.make_query(B, Hq, d, seed=11)
    key, value, kn, avg = synth.make_kv(B, Hkv, n, d, seed=12, dist="gauss")
    ref = run_reference_chain(B, Hq, Hkv, d, K, L, n, M, key, value, kn, hf, q)
    # nnz = 0 edge: a query whose codes are all NB-1 XOR the majority never collides twice
    # (constructed: use codes no key carries in that table)
    kc = torch.from_numpy(ref["kcodes"])  # (B,Hkv,L,n)
    miss = torch.zeros((B * Hq, L), dtype=torch.int32)
    for h in range(B * Hq):
        b, g = h // Hq, (h % Hq) // (Hq // Hkv)
        for l in range(L):
            present = set(kc[b, g, l].tolist())
            miss[h, l] = next(c for c in range(1 << K) if c not in present)
    ref0 = run_reference_chain(B, Hq, Hkv, d, K, L, n, M, key, value, kn, hf, q, qcodes=miss)
    assert int(ref0["nnz"].sum()) == 0
    np.savez_compressed(
        os.path.join(HERE, "small_chain.npz"),
        dims=np.array([B, Hq, Hkv, d, K, L, n, M]), hash_func=u16(hf), query=u16(q), key=u16(key), value=u16(value),
        key_norm=kn.numpy(), avg_k=u16(avg), miss_qcodes=miss.numpy(), miss_nnz=ref0["nnz"], miss_out_bf16=ref0["out_bf16"],
        miss_lse2=ref0["mve"][1], **ref)
    print("small_chain: nnz", ref["nnz"].tolist())


def make_c1():
    B, Hq, Hkv, d, K, L, n = 1, 1, 1, 128, 10, 150, 4096
    M = n + 128
    hf = synth.make_hash_func(d, K, L, seed=0)
    q = synth.make_query(B, Hq, d, seed=1)
    key, value, kn, avg = synth.make_kv(B, Hkv, n, d, seed=2, dist="clustered", q_dirs=q.reshape(B, Hq, d)[:, :1].float())
    ref = run_reference_chain(B, Hq, Hkv, d, K, L, n, M, key, value, kn, hf, q)
    ref.pop("kcodes")
    ref.pop("mask")
    np.savez_compressed(os.path.join(HERE, "c1_chain.npz"), dims=np.array([B, Hq, Hkv, d, K, L, n, M]),
                        input_sha256=np.array(checksum(hf, q, key, value, kn)), **ref)
    print("c1_chain: nnz", ref["nnz"].tolist(), "sha", checksum(hf, q, key, value, kn)[:16])


def probe_case_inputs(K, L, seq, delta, group, bsz):
    """Seeded inputs of one probe case: key codes (bsz, Hkv, L, seq) int16 and query codes (bsz*Hq, L) int32."""
    g = torch.Generator().manual_seed(K * 1000 + L)
    Hq = 32
    codes = torch.randint(0, 1 << K, (bsz, Hq // group, L, seq), generator=g, dtype=torch.int16)
    query = torch.randint(0, 1 << K, (bsz * Hq, L), generator=g, dtype=torch.int32)
    return codes, query


def probe_case_key(K, L, seq, delta, group, bsz) -> str:
    return f"probe_K{K}_L{L}_seq{seq}_delta{delta}_group{group}_bsz{bsz}"


ATTN_DIMS = dict(B=1, Hq=8, Hkv=2, d=128, K=10, L=150, n=2048, M=2048 + 128)


def attention_case_inputs():
    """Seeded inputs of the attention case: key/value (B,Hkv,n,d) bf16, their norms, queries (B*Hq,d) bf16, nnz and index
    sets (B*Hq, M) int32."""
    B, Hq, Hkv, d, n, M = (ATTN_DIMS[k] for k in ("B", "Hq", "Hkv", "d", "n", "M"))
    g = torch.Generator().manual_seed(77)
    key = torch.randn((B, Hkv, n, d), generator=g).bfloat16()
    value = torch.randn((B, Hkv, n, d), generator=g).bfloat16()
    kn = key.norm(p=2, dim=-1).float()
    q = torch.randn((B * Hq, d), generator=g).bfloat16()
    nnz = torch.randint(1, n, (B * Hq,), generator=g).int()
    ind = torch.zeros((B * Hq, M), dtype=torch.int32)
    for h in range(B * Hq):
        ind[h, : nnz[h]] = torch.randperm(n, generator=g)[: nnz[h]].int()
    return key, value, kn, q, nnz, ind


def make_operator_cases():
    lsh_m, sa_m, flavour = ref_loader.load()
    out = {"flavour": np.array(flavour)}
    for case in PROBE_CASES:
        K, L, seq, delta, group, bsz = case
        Hq, M = 32, seq + delta
        codes, query = probe_case_inputs(*case)
        sc, si = codes.sort()
        R = lsh_m.LSH()
        R.alloc(K, L, 1, Hq, Hq // group, bsz, M)
        for b in range(bsz):
            R.fill(0, b, sc[b].contiguous(), si[b].int().contiguous())
        results = torch.zeros((bsz * Hq, M), dtype=torch.int32)
        nnz = torch.zeros((bsz * Hq,), dtype=torch.int32)
        R.batch_retrieve(0, query, results, nnz)
        mask = R.get_mask().clone().view(torch.uint8).reshape(bsz * Hq, M)
        k = probe_case_key(*case)
        out.update({f"{k}_input_sha256": np.array(checksum(codes, query)), f"{k}_nnz": nnz.numpy(), f"{k}_results": results.numpy(),
                    f"{k}_mask": mask.numpy()})
    B, Hq, Hkv, d, K, L, M = (ATTN_DIMS[k] for k in ("B", "Hq", "Hkv", "d", "K", "L", "M"))
    key, value, kn, q, nnz, ind = attention_case_inputs()
    S = sa_m.SparseAttentionServer()
    S.alloc(1, Hq, Hkv, d, B, M)
    S.fill(0, 0, key[0].contiguous(), value[0].contiguous(), kn[0].contiguous())
    o = torch.zeros((B * Hq, d), dtype=torch.bfloat16)
    mve = torch.zeros((2, B * Hq))
    S.attention_wrapper(0, K, L, o, mve, q, q.float().norm(p=2, dim=-1), ind, nnz)
    out.update({"attn_input_sha256": np.array(checksum(key, value, kn, q, nnz, ind)), "attn_out_bf16": u16(o), "attn_mve": mve.numpy()})
    np.savez_compressed(os.path.join(HERE, "operator_cases.npz"), **out)
    print("operator_cases:", {probe_case_key(*c): int(out[probe_case_key(*c) + "_nnz"].sum()) for c in PROBE_CASES})


def _calls(tree, want):
    """Every call `want(node)` names, as {"method", "n_args", "keywords"} (a keyword of None stands for **kwargs)."""
    out = []
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and (m := want(node)):
            out.append({**m, "n_args": len(node.args), "keywords": [k.arg for k in node.keywords]})
    return out


def make_reference_api():
    from oracle.build_ref import REF

    def parse(path):
        with open(os.path.join(REF, path)) as f:
            return ast.parse(f.read())

    def cls_node(tree, name):
        return next(n for n in ast.walk(tree) if isinstance(n, ast.ClassDef) and n.name == name)

    server = cls_node(parse("models/attnserver.py"), "LSHSparseAttnServer")
    methods = {}
    for fn in server.body:
        if not isinstance(fn, ast.FunctionDef):
            continue
        args = [a.arg for a in fn.args.args]
        defaults = []
        for a, dflt in zip(args[len(args) - len(fn.args.defaults):], fn.args.defaults):
            try:
                defaults.append({"arg": a, "literal": True, "value": ast.literal_eval(dflt)})
            except ValueError:
                defaults.append({"arg": a, "literal": False, "value": None})   # e.g. torch.bfloat16
        methods[fn.name] = {"args": args, "defaults": defaults}

    def llama_call(node):   # llama.py:92-93 constructor, self.attention_server.<method>(...) elsewhere
        f = node.func
        if isinstance(f, ast.Name) and f.id == "LSHSparseAttnServer":
            return {"method": "__init__"}
        if isinstance(f, ast.Attribute) and isinstance(f.value, ast.Attribute) and f.value.attr == "attention_server":
            return {"method": f.attr}
        return None

    def operator_call(node):   # self.attn_server.<method>(...) / self.lsh_retriever.<method>(...)
        f = node.func
        if isinstance(f, ast.Attribute) and isinstance(f.value, ast.Attribute) and f.value.attr in ("attn_server", "lsh_retriever"):
            return {"owner": f.value.attr, "method": f.attr}
        return None

    def pybind_defs(path):
        with open(os.path.join(REF, path)) as f:
            return re.findall(r'\.def\("([a-z_0-9]+)"', f.read())

    def cpp_members(path, cls):
        """method name -> parameter names (without the `_pt` suffix the reference gives tensor arguments)."""
        with open(os.path.join(REF, path)) as f:
            text = f.read()
        body = text[text.index(f"class {cls}"):]
        body = body[: body.index("private:")]
        out = {}
        for m in re.finditer(r"(?:void|torch::Tensor|int)\s+([a-z_0-9]+)\(([^)]*)\);", body):
            params = [p.strip().split()[-1] for p in m.group(2).split(",") if p.strip()]
            out[m.group(1)] = [re.sub(r"_pt$", "", p) for p in params]
        return out

    api = {
        "attnserver_methods": methods,
        "llama_calls": _calls(parse("models/llama.py"), llama_call),
        "attnserver_operator_calls": _calls(server, operator_call),
        "pybind_defs": {p: pybind_defs(p) for p in ("library/lsh/lsh.cc", "library/sparse_attention/sparse_attention.cc")},
        "cpp_members": {"library/lsh/lsh.h": {"LSH": cpp_members("library/lsh/lsh.h", "LSH")},
                        "library/sparse_attention/sparse_attention.h":
                            {"SparseAttentionServer": cpp_members("library/sparse_attention/sparse_attention.h", "SparseAttentionServer")}},
    }
    with open(os.path.join(HERE, "reference_api.json"), "w") as f:
        json.dump(api, f, indent=1, sort_keys=True)
        f.write("\n")
    print("reference_api:", {k: len(v) for k, v in api.items()})


if __name__ == "__main__":
    torch.set_num_threads(4)
    make_small()
    make_c1()
    make_operator_cases()
    make_reference_api()
