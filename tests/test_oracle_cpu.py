"""CPU suite (`-m "not gpu"`): pins the oracle and checks the host-side plumbing.

  * oracle/mpig_oracle.c (the C restatement) against the committed golden vectors produced by the
    reference's own compiled operators (tests/golden/make_golden.py);
  * the selection rule and the attention math against the reference tests' torch formulas
    (library/lsh/test.py:43, library/sparse_attention/test_sparse.py:68-84);
  * the C-ABI shared library loads and exports every symbol include/magicpig_b200.h declares.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

import oracle
from magicpig_b200 import synth, _native
from tests.golden.make_golden import ATTN_DIMS, PROBE_CASES, attention_case_inputs, checksum, probe_case_inputs, probe_case_key

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def bf16_from_u16(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(a.view(np.int16).copy()).view(torch.bfloat16)


def load_small():
    z = np.load(os.path.join(GOLD, "small_chain.npz"))
    B, Hq, Hkv, d, K, L, n, M = [int(x) for x in z["dims"]]
    t = dict(B=B, Hq=Hq, Hkv=Hkv, d=d, K=K, L=L, n=n, M=M)
    t["hash_func"] = bf16_from_u16(z["hash_func"]).reshape(d, K * L)
    t["query"] = bf16_from_u16(z["query"]).reshape(B, Hq, 1, d)
    t["key"] = bf16_from_u16(z["key"]).reshape(B, Hkv, n, d)
    t["value"] = bf16_from_u16(z["value"]).reshape(B, Hkv, n, d)
    t["key_norm"] = torch.from_numpy(z["key_norm"])
    t["avg_k"] = bf16_from_u16(z["avg_k"]).reshape(B, Hkv, 1, d)
    for k in ("kcodes", "qcodes", "nnz", "results_sorted", "results_offsets", "mask", "mve", "miss_qcodes", "miss_nnz",
              "miss_lse2"):
        t[k] = torch.from_numpy(z[k])
    t["out"] = bf16_from_u16(z["out_bf16"]).reshape(B * Hq, d)
    t["miss_out"] = bf16_from_u16(z["miss_out_bf16"]).reshape(B * Hq, d)
    return t


def pad_store(t):
    """(B,Hkv,n,d) -> reference-shaped (B*Hkv, M, d) stores."""
    B, Hkv, n, d, M = t["B"], t["Hkv"], t["n"], t["d"], t["M"]
    k = torch.zeros((B * Hkv, M, d), dtype=torch.bfloat16)
    v = torch.zeros((B * Hkv, M, d), dtype=torch.bfloat16)
    kn = torch.zeros((B * Hkv, M), dtype=torch.float32)
    k[:, :n] = t["key"].reshape(B * Hkv, n, d)
    v[:, :n] = t["value"].reshape(B * Hkv, n, d)
    kn[:, :n] = t["key_norm"].reshape(B * Hkv, n)
    return k, v, kn


def port_probe(t, qcodes):
    """oracle port over all requests -> results (H,M), nnz (H), mask (H,M)."""
    B, Hq, Hkv, K, L, M = t["B"], t["Hq"], t["Hkv"], t["K"], t["L"], t["M"]
    G = Hq // Hkv
    res, nz, mk = [], [], []
    sc, si = t["kcodes"].sort()
    for b in range(B):
        T = oracle.Tables(Hkv, L, K, M)
        T.fill(sc[b].contiguous(), si[b].int().contiguous())
        r, n_, m_ = oracle.batch_retrieve(T, qcodes[b * Hq:(b + 1) * Hq].contiguous(), G)
        res.append(r), nz.append(n_), mk.append(m_)
    return torch.cat(res), torch.cat(nz), torch.cat(mk)


def test_port_probe_matches_golden():
    t = load_small()
    res, nnz, mask = port_probe(t, t["qcodes"])
    assert torch.equal(nnz, t["nnz"])
    assert torch.equal(mask, t["mask"])
    offs = t["results_offsets"]
    for h in range(t["B"] * t["Hq"]):
        mine = res[h, : nnz[h]].sort().values
        assert torch.equal(mine, t["results_sorted"][offs[h]:offs[h + 1]])
    # and the selection rule itself (library/lsh/test.py:43)
    for b in range(t["B"]):
        cnt = oracle.collision_counts(t["kcodes"][b].contiguous(), t["qcodes"][b * t["Hq"]:(b + 1) * t["Hq"]].contiguous(),
                                      t["Hq"] // t["Hkv"])
        assert torch.equal((cnt > 1).sum(-1).int(), nnz[b * t["Hq"]:(b + 1) * t["Hq"]])
        assert torch.equal(cnt.clamp(max=2).to(torch.uint8), mask[b * t["Hq"]:(b + 1) * t["Hq"], : t["n"]])


def test_port_attention_matches_golden():
    t = load_small()
    res, nnz, _ = port_probe(t, t["qcodes"])
    k, v, kn = pad_store(t)
    q = t["query"].reshape(-1, t["d"])
    qn = q.float().norm(p=2, dim=-1)
    out, mve, _ = oracle.attention_wrapper(k, v, kn, t["K"], t["L"], q, qn, res, nnz)
    # reference's own tolerance for this operator is 1e-2 (test_sparse.py:87,92)
    assert torch.allclose(out.float(), t["out"].float(), rtol=1e-2, atol=1e-2)
    assert torch.allclose(mve[1], t["mve"][1], atol=2e-2), (mve[1], t["mve"][1])


def test_port_nnz0_edge_matches_golden():
    t = load_small()
    res, nnz, _ = port_probe(t, t["miss_qcodes"])
    assert int(nnz.sum()) == 0 and int(t["miss_nnz"].sum()) == 0
    k, v, kn = pad_store(t)
    q = t["query"].reshape(-1, t["d"])
    out, mve, _ = oracle.attention_wrapper(k, v, kn, t["K"], t["L"], q, q.float().norm(p=2, dim=-1), res, nnz)
    assert torch.equal(out.float(), torch.zeros_like(out.float())) and torch.equal(t["miss_out"].float(), out.float())
    assert torch.isinf(mve[1]).all() and (mve[1] < 0).all()
    assert torch.isinf(t["miss_lse2"]).all() and (t["miss_lse2"] < 0).all()


def test_port_c1_matches_golden():
    """BASELINE config[0]: 1 head, seq 4096, d 128, K10 L150 -- inputs regenerated from seeds."""
    z = np.load(os.path.join(GOLD, "c1_chain.npz"))
    B, Hq, Hkv, d, K, L, n, M = [int(x) for x in z["dims"]]
    hf = synth.make_hash_func(d, K, L, seed=0)
    q = synth.make_query(B, Hq, d, seed=1)
    key, value, kn, _ = synth.make_kv(B, Hkv, n, d, seed=2, dist="clustered", q_dirs=q.reshape(B, Hq, d)[:, :1].float())
    from tests.golden.make_golden import checksum
    if checksum(hf, q, key, value, kn) != str(z["input_sha256"]):
        pytest.skip("torch RNG stream differs from the one that produced the fixture")
    kcodes = synth.hash_keys(key, hf, K, L)
    qcodes = synth.hash_queries_ref(q, hf, K, L)
    assert torch.equal(qcodes, torch.from_numpy(z["qcodes"]))
    pq, margin = oracle.simhash(q.reshape(-1, d), hf, K, L)
    assert (pq != qcodes).sum() == 0 or margin[pq != qcodes].max() < 1e-3
    t = dict(B=B, Hq=Hq, Hkv=Hkv, d=d, K=K, L=L, n=n, M=M, kcodes=kcodes, key=key, value=value, key_norm=kn)
    res, nnz, _ = port_probe(t, qcodes)
    assert torch.equal(nnz, torch.from_numpy(z["nnz"]))
    assert torch.equal(res[0, : nnz[0]].sort().values, torch.from_numpy(z["results_sorted"]))
    k, v, knp = pad_store(t)
    q2 = q.reshape(-1, d)
    out, mve, _ = oracle.attention_wrapper(k, v, knp, K, L, q2, q2.float().norm(p=2, dim=-1), res, nnz)
    ref_out = bf16_from_u16(z["out_bf16"]).reshape(1, d)
    assert torch.allclose(out.float(), ref_out.float(), rtol=1e-2, atol=1e-2)
    assert abs(float(mve[1, 0]) - float(z["mve"][1, 0])) < 2e-2


def test_port_attention_vs_torch_formula():
    """Appendix A in fp64 (= test_sparse.py:68-84) vs the C restatement, random index sets."""
    torch.manual_seed(3)
    BHkv, G, n, d, K, L = 2, 4, 512, 128, 10, 150
    H = BHkv * G
    key = torch.randn(BHkv, n, d).bfloat16()
    value = torch.randn(BHkv, n, d).bfloat16()
    kn = key.norm(p=2, dim=-1).float()
    q = torch.randn(H, d).bfloat16()
    nnz = torch.randint(1, n, (H,)).int()
    ind = torch.zeros((H, n), dtype=torch.int32)
    sets = []
    for h in range(H):
        s = torch.randperm(n)[: nnz[h]].int()
        ind[h, : nnz[h]] = s
        sets.append(s)
    out, mve, score = oracle.attention_wrapper(key, value, kn, K, L, q, q.float().norm(p=2, dim=-1), ind, nnz, want_score=True)
    ref_out, ref_lse = synth.torch_reference_attention(key, value, kn, q, sets, K, L, G)
    assert torch.allclose(out.double(), ref_out, rtol=1e-2, atol=4e-3)  # bf16 output rounding dominates
    assert torch.allclose(mve[1].double(), ref_lse, atol=1e-3)
    for h in range(H):
        assert abs(float(score[h, : nnz[h]].sum()) - 1) < 1e-4
        # the error budget the GPU suite applies (tests/test_gpu_parity.py::assert_1e3_before_rounding) holds for the port's
        # own bf16 output against its un-rounded value sum_j p_j V_j: half a bf16 ulp + 1e-3 of the largest element
        o_pre = score[h, : nnz[h]].double() @ value[h // G][sets[h].long()].double()
        budget = o_pre.abs() * 2.0 ** -8 + 1e-3 * o_pre.abs().max()
        assert bool(((out[h].double() - o_pre).abs() <= budget).all())


def test_port_simhash_vs_torch():
    torch.manual_seed(5)
    d, K, L, H = 128, 10, 150, 32
    hf = synth.make_hash_func(d, K, L, seed=7)
    q = synth.make_query(1, H, d, seed=8).reshape(H, d)
    codes, margin = oracle.simhash(q, hf, K, L)
    ref = synth.hash_queries_ref(q, hf, K, L)
    bad = codes != ref
    assert bad.sum() == 0 or float(margin[bad].max()) < 1e-3


def test_window_and_merge_restatement():
    """merge(window, sparse) == softmax over the union (the identity the fused kernel relies on)."""
    torch.manual_seed(9)
    d, w, n, G = 128, 37, 200, 1
    kw = torch.randn(1, w, d).bfloat16()
    vw = torch.randn(1, w, d).bfloat16()
    q = torch.randn(1, d).bfloat16()
    o_w, lse_w = oracle.window_attention(kw, vw, q, G)
    s = (kw[0].double() @ q[0].double()) / np.sqrt(d)
    p = torch.softmax(s, 0)
    assert torch.allclose(o_w[0].double(), p @ vw[0].double(), atol=1e-5)
    assert abs(float(lse_w[0]) - float(torch.logsumexp(s, 0) / np.log(2))) < 1e-4
    k2 = torch.randn(1, n, d).bfloat16()
    v2 = torch.randn(1, n, d).bfloat16()
    o2, lse2 = oracle.window_attention(k2, v2, q, G)
    om, lm = oracle.merge_state(o_w, lse_w, o2, lse2)
    ou, lu = oracle.window_attention(torch.cat([kw, k2], 1), torch.cat([vw, v2], 1), q, G)
    assert torch.allclose(om, ou, atol=1e-5) and abs(float(lm[0] - lu[0])) < 1e-4


def load_operator_case(key: str, *inputs):
    """The compiled reference's outputs for one case of operator_cases.npz, after checking that the seeded inputs are the
    ones they were computed from."""
    z = np.load(os.path.join(GOLD, "operator_cases.npz"))
    assert checksum(*inputs) == str(z[f"{key}_input_sha256"]), "inputs differ from the ones the stored reference outputs belong to"
    return {k[len(key) + 1:]: z[k] for k in z.files if k.startswith(key + "_")}


@pytest.mark.parametrize("K,L,seq,delta,group,bsz", PROBE_CASES)
def test_port_probe_vs_live_reference(K, L, seq, delta, group, bsz):
    """library/lsh/test.py's own case shape, checked three ways: the reference binary's recorded outputs
    (tests/golden/operator_cases.npz), port, torch formula."""
    Hq = 32
    Hkv = Hq // group
    M = seq + delta
    codes, query = probe_case_inputs(K, L, seq, delta, group, bsz)
    ref = load_operator_case(probe_case_key(K, L, seq, delta, group, bsz), codes, query)
    results, nnz, mask = (torch.from_numpy(ref[k]) for k in ("results", "nnz", "mask"))
    assert results.shape == mask.shape == (bsz * Hq, M)
    sc, si = codes.sort()
    for b in range(bsz):
        T = oracle.Tables(Hkv, L, K, M)
        T.fill(sc[b].contiguous(), si[b].int().contiguous())
        r, nz, mk = oracle.batch_retrieve(T, query[b * Hq:(b + 1) * Hq].contiguous(), group)
        sl = slice(b * Hq, (b + 1) * Hq)
        assert torch.equal(nz, nnz[sl]) and torch.equal(r, results[sl]) and torch.equal(mk, mask[sl])
        cnt = oracle.collision_counts(codes[b].contiguous(), query[sl].contiguous(), group)
        assert torch.equal((cnt > 1).sum(-1).int(), nz)


def test_port_attention_vs_live_reference():
    """SparseAttentionServer.attention_wrapper's recorded outputs (tests/golden/operator_cases.npz) vs the port."""
    B, Hq, Hkv, d, K, L, n, M = (ATTN_DIMS[k] for k in ("B", "Hq", "Hkv", "d", "K", "L", "n", "M"))
    key, value, kn, q, nnz, ind = attention_case_inputs()
    ref = load_operator_case("attn", key, value, kn, q, nnz, ind)
    out_ref = bf16_from_u16(ref["out_bf16"]).reshape(B * Hq, d)
    mve_ref = torch.from_numpy(ref["mve"])
    qn = q.float().norm(p=2, dim=-1)
    t = dict(B=B, Hkv=Hkv, n=n, d=d, M=M, key=key, value=value, key_norm=kn)
    k, v, knp = pad_store(t)
    out, mve, _ = oracle.attention_wrapper(k, v, knp, K, L, q, qn, ind, nnz)
    assert torch.allclose(out.float(), out_ref.float(), rtol=1e-2, atol=1e-2)
    assert torch.allclose(mve[1], mve_ref[1], atol=2e-2)


# ------------------------------------------------------------------------------------------------
# C-ABI library: builds, loads, exports everything the header declares.  No compute without a GPU.
# ------------------------------------------------------------------------------------------------
def test_cabi_exports_every_declared_symbol():
    from magicpig_b200 import build
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    declared = _native.declared_symbols()
    assert len(declared) >= 20
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, f"header declares symbols the library does not export: {missing}"
    assert set(declared) == set(_native._SIGNATURES), "ctypes signature table out of sync with the header"
    aux = _native.declared_symbols(_native.AUX_HEADER_PATH)       # include/magicpig_b200_aux.h: harness-side helpers
    assert len(aux) >= 5
    assert not [s for s in aux if not hasattr(lib, s)], "aux header declares symbols the library does not export"
    assert set(aux) == set(_native._AUX_SIGNATURES), "ctypes signature table out of sync with the aux header"
    lib.mpig_abi_version.restype = ctypes.c_int
    assert lib.mpig_abi_version() == _native.MPIG_ABI_VERSION


def test_no_cpu_fallback():
    """The product fails loudly without a CUDA device instead of computing somewhere else."""
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from magicpig_b200.ops import Context
    with pytest.raises(Exception):
        Context(10, 150, 1, 32, 8, 128, 1, 4096, device="cpu")
    with pytest.raises(Exception):
        Context(10, 150, 1, 32, 8, 128, 1, 4096, device="cuda:0")


def test_product_does_not_import_oracle():
    root = os.path.join(os.path.dirname(os.path.dirname(__file__)), "magicpig_b200")
    for dp, _, files in os.walk(root):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "oracle/" not in src.replace("oracle/_ref", ""), f
