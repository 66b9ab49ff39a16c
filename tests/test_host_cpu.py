"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host logic,
impression sharding over gloo (world_size 2).  No compute calls (there is no GPU here)."""
import os
import re
import socket

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "nrb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nrb_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_loads_and_exports_every_symbol():
    from news_recommendation_project_v2_b200 import _lib, build
    build.build()
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/nrb200.h but not exported"
        assert n in _lib.PROTOTYPES, f"{n} has no ctypes prototype"
    assert set(_lib.PROTOTYPES) == set(names)
    assert b"sm_100a" in lib.nrb_version()


def test_no_cpu_fallback_without_gpu():
    from news_recommendation_project_v2_b200 import _lib
    from news_recommendation_project_v2_b200.data_utils import rank_group_preds
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.NrbError):
        rank_group_preds(np.array([1.0, 2.0], dtype=np.float32), np.array([2], dtype=np.int32))
    m = LatentAttentionModel(dim=64, num_latents=32, heads=2, dim_head=32).eval()
    with pytest.raises(_lib.NrbError):
        m(torch.zeros(1, 4, 64), torch.ones(1, 4, dtype=torch.int32))
    assert _lib.load().nrb_check_device(0) != 0 and b"no CUDA device" in _lib.load().nrb_last_error()


def test_argument_validation_without_gpu():
    """Bad shapes are rejected by the library before any CUDA call."""
    from news_recommendation_project_v2_b200 import _lib
    lib = _lib.load()
    rc = lib.nrb_score_rank(0, 1, 100, 10, 1, 1, 100, 1, 100, None, 1.0, 1, 1, 1, 1, 4, None, 1, None, 1, None)
    assert rc == -1 and b"multiple of 512" in lib.nrb_last_error()
    rc = lib.nrb_score_rank(7, 1, 256, 10, 1, 1, 256, 1, 256, None, 1.0, 1, 1, 1, 1, 4, None, 1, None, 1, None)
    assert rc == -1 and b"pool_mode" in lib.nrb_last_error()
    assert lib.nrb_dense_rank(None, None, 0, None, None) == 0  # empty problem is a no-op
    assert lib.nrb_dense_rank_f64(None, None, 0, None, None) == 0
    assert lib.nrb_final_attention_rows_workspace_bytes(1, 161013, 1024, 4096) > 2 * 16384 * 4096 * 2
    # round-2 entry points
    assert lib.nrb_final_attention_rows_split_workspace_bytes(161013, 1024, 4096) >= 16384 * 4096 * (4 + 6)
    assert lib.nrb_split_rows(1, 1024, 1, 3072, 8, 1022, 0, None) == -1 and b"multiple of 4" in lib.nrb_last_error()
    assert lib.nrb_split_rows(1, 1024, 1, 3072, 8, 1024, 5, None) == -1 and b"role" in lib.nrb_last_error()
    assert lib.nrb_convert_rows(1, 7, 8, 1, 1, 8, 4, 8, None) == -1 and b"dtype" in lib.nrb_last_error()
    assert lib.nrb_narrow_ranks(None, None, 0, None, None) == 0
    assert lib.nrb_narrow_ranks(4, 8, 16, 12, None) == -1 and b"aligned" in lib.nrb_last_error()
    assert lib.nrb_mask_to_csr(None, -1, 4, None, None, None, None) == -1
    assert lib.nrb_push_attach(None, 4, 1) == -1 and b"at most" in lib.nrb_last_error()
    assert lib.nrb_push_attach(None, 0, 0) == -1 and b"spread" in lib.nrb_last_error()
    lib.nrb_push_cancel()
    assert lib.nrb_push_flush(None) == 0  # nothing pending: no launch, no CUDA call
    # latent fold: any latent count passes the size checks (here it stops at the null pointers); bf16 with
    # heads * latents_padded not a multiple of 64 is refused by name, in the library and before any device work in ops
    assert lib.nrb_latent_fold(0, 64, 2, 32, 50, *[None] * 9, 0, None) == -1 and b"null" in lib.nrb_last_error()
    assert lib.nrb_latent_fold(1, 64, 1, 32, 409, *[None] * 9, 0, None) == -1 and b"null" in lib.nrb_last_error()
    assert lib.nrb_latent_fold(1, 64, 1, 32, 32, *[None] * 9, 0, None) == -1
    assert b"heads * latents_padded" in lib.nrb_last_error() and b"1 x 32" in lib.nrb_last_error()
    # (the fold's FFMA GEMMs run over the latent count rounded up to a multiple of 4)
    assert lib.nrb_latent_fold_workspace_bytes(64, 2, 32, 50) == lib.nrb_latent_fold_workspace_bytes(64, 2, 32, 52)
    from news_recommendation_project_v2_b200 import ops, synthetic as syn
    sd = syn.make_latent_state_dict(64, 20, heads=3, dim_head=32, seed=0)
    with pytest.raises(_lib.NrbError, match=r"heads \* latents_padded .*\(got 3 x 32\)"):
        ops.latent_fold(sd, 3, 32, torch.bfloat16, None)


def test_host_copy_is_exact_for_any_thread_count():
    """nrb_host_copy (page cache -> pinned staging of the packed token file) is a plain byte copy."""
    from news_recommendation_project_v2_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(0)
    for n in (0, 1, 4095, 3 * (1 << 20) + 17, 9 * (1 << 20)):
        src = rng.integers(0, 256, size=n, dtype=np.uint8)
        for nt in (1, 3, 8):
            dst = np.full(n + 8, 0xAB, dtype=np.uint8)
            assert lib.nrb_host_copy(dst.ctypes.data if n else None, src.ctypes.data if n else None, n, nt) == 0
            assert np.array_equal(dst[:n], src) and (dst[n:] == 0xAB).all()
    assert lib.nrb_host_copy(None, None, 8, 2) == -1


def test_state_dict_keys_match_reference(golden_dir):
    from news_recommendation_project_v2_b200.latent_attention import LatentAttentionModel
    from news_recommendation_project_v2_b200.modeling_utils import FinalAttention
    g = np.load(os.path.join(golden_dir, "latent_cfg1_d768_L512.npz"))
    m = LatentAttentionModel(dim=768, num_latents=512)
    sd = m.state_dict()
    assert sorted(sd) == list(g["keys"])
    assert [str(tuple(sd[k].shape)) for k in sorted(sd)] == list(g["shapes"])
    # reference defaults: 64 latents, 8 heads x 512, dim from the config global (latent_attention.py:99-104)
    d = LatentAttentionModel()
    assert d.latents.shape == (64, 1024) and d.cross_attend_blocks[0].fn.to_q.weight.shape == (4096, 1024)
    fa = FinalAttention(768, 4096)
    assert sorted(fa.state_dict()) == sorted(
        [f"linear{i}.weight" for i in range(1, 6)] + [f"linear{i}.bias" for i in range(1, 5)])


def test_reference_checkpoints_load_through_the_factories(golden_dir, tmp_path, monkeypatch):
    """torch.save(state_dict in the reference's layout) -> get_*_model(path) (modeling_utils.py:151-155, 274-279):
    strict load, every tensor identical, eval mode.  The checkpoints are the synthetic weights that the reference's own
    modules loaded strictly when the golden vectors were minted (oracle/make_golden.py), pinned by the weight digests
    stored with those vectors."""
    from news_recommendation_project_v2_b200 import config, modeling_utils as mu, synthetic as syn
    from oracle.make_golden import sd_digest
    monkeypatch.setattr(config, "DEVICE", torch.device("cpu"))
    for name, factory in (("final_small_d768", mu.get_final_attention_model),
                          ("final_large_d1024", mu.get_final_attention_model),
                          ("latent_default_d1024_L64", mu.get_latent_attention_model)):
        g = np.load(os.path.join(golden_dir, name + ".npz"))
        dim, seed = int(g["dim"]), int(g["seed"])
        monkeypatch.setattr(config, "REDUCED_DIM", dim)
        monkeypatch.setattr(config, "EMBEDDING_DIM", dim)
        if factory is mu.get_final_attention_model:
            sd = syn.make_final_attention_state_dict(dim, int(g["hidden"]), seed=seed)
        else:
            sd = syn.make_latent_state_dict(dim, int(g["L"]), seed=seed)
            assert sorted(sd) == list(g["keys"])
        assert sd_digest(sd) == str(g["sd_sha256"]), name
        p = tmp_path / f"{name}.pt"
        torch.save(sd, p)
        ours = factory(p)
        assert not ours.training and set(ours.state_dict()) == set(sd)
        for k, v in sd.items():
            assert torch.equal(ours.state_dict()[k], v), k
    with pytest.raises(RuntimeError):
        mu.get_latent_attention_model(tmp_path / "final_large_d1024.pt")  # wrong architecture: strict load refuses


def test_group_items_pad_and_rank_object_arrays():
    from news_recommendation_project_v2_b200.data_utils import group_items, pad_to_maxlen, ranks_to_object_array
    items = np.arange(10, dtype=np.int32)
    g = group_items(items, np.array([3, 0, 7], dtype=np.int32))
    assert g.dtype == object and [list(x) for x in g] == [[0, 1, 2], [], [3, 4, 5, 6, 7, 8, 9]]
    # equal counts stay a 1-D object array (the reference's version turns 2-D and crashes later: quirk a7)
    g2 = group_items(items[:6], np.array([3, 3], dtype=np.int32))
    assert g2.shape == (2,) and g2.dtype == object
    p = pad_to_maxlen([np.array([5, 6], dtype=np.int32), np.array([7], dtype=np.int32)])
    assert p["indices"].tolist() == [[5, 6], [7, 0]] and p["attention_mask"].tolist() == [[1, 1], [1, 0]]
    assert p["indices"].dtype == np.int32 and p["attention_mask"].dtype == np.int32
    r = ranks_to_object_array(np.array([1, 2, 0, 0], dtype=np.int32), np.array([2, 2], dtype=np.int32))
    assert r[0].tolist() == [1.0, 2.0] and np.isnan(r[1]).all() and r[0].dtype == np.float32


def test_partition_is_contiguous_and_balanced():
    from news_recommendation_project_v2_b200 import synthetic as syn
    from news_recommendation_project_v2_b200.sharding import partition_impressions, shard_impressions
    imp = syn.make_impressions(5000, 1000, cand="large", seed=1)
    for world in (1, 2, 3, 8):
        parts = partition_impressions(imp.hist_len, imp.cand_len, world)
        assert parts[0][0] == 0 and parts[-1][1] == imp.n
        assert all(parts[i][1] == parts[i + 1][0] for i in range(world - 1))
        cost = 2 * imp.hist_len.astype(np.int64) + imp.cand_len
        loads = [cost[a:b].sum() for a, b in parts]
        assert max(loads) <= 1.02 * cost.sum() / world + cost.max()
    a, b = partition_impressions(imp.hist_len, imp.cand_len, 2)[1]
    hi, hl, ci, cl = shard_impressions(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, a, b)
    assert hi.shape[0] == hl.sum() and ci.shape[0] == cl.sum()
    assert np.array_equal(ci, imp.cand_idx[imp.cand_len[:a].sum():])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    from news_recommendation_project_v2_b200 import synthetic as syn
    from news_recommendation_project_v2_b200.sharding import (gather_ordered, partition_impressions, reduce_sums,
                                                              shard_impressions)
    from oracle import oracle
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        imp = syn.make_impressions(64, 200, h_max=9, seed=3)
        rng = np.random.default_rng(0)
        all_scores = rng.standard_normal(int(imp.cand_len.sum())).astype(np.float32)
        a, b = partition_impressions(imp.hist_len, imp.cand_len, world)[rank]
        _, _, _, cl = shard_impressions(imp.hist_idx, imp.hist_len, imp.cand_idx, imp.cand_len, a, b)
        c_off = syn.csr_offsets(imp.cand_len)
        local_scores = all_scores[c_off[a]:c_off[b]]
        # each rank "scores" its block (here: dense ranks by the oracle), then ordered gather
        local_ranks = np.concatenate(oracle.rank_group_preds(local_scores, cl) + [np.zeros(0)]).astype(np.int32)
        ranks = gather_ordered(torch.from_numpy(local_ranks))
        sums = reduce_sums([float(local_ranks.sum()), float(len(cl))])
        want = np.concatenate(oracle.rank_group_preds(all_scores, imp.cand_len)).astype(np.int32)
        ok = np.array_equal(ranks.numpy(), want) and sums == [float(want.sum()), float(imp.n)]
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_sharded_gather_gloo_world2():
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_gloo_worker, args=(world, port, out), nprocs=world, join=True)
        assert dict(out) == {0: True, 1: True}


def test_table_shard_bounds():
    from news_recommendation_project_v2_b200.sharding import table_shard_bounds
    b = table_shard_bounds(10_000_000, 8)
    assert b[0] == (0, 1_250_000) and b[-1] == (8_750_000, 10_000_000)
    b = table_shard_bounds(40_003, 2)
    assert b == [(0, 20_002), (20_002, 40_003)]
    b = table_shard_bounds(5, 8)  # more ranks than rows: trailing shards are empty
    assert b[:5] == [(i, i + 1) for i in range(5)] and all(x == (5, 5) for x in b[5:])


def test_native_csr_builder_matches_reference(golden_dir):
    """nrb_csr_build (host C++) vs the reference's split_impressions_and_history golden + a random log."""
    from news_recommendation_project_v2_b200.data_utils import split_impressions_and_history
    from oracle import oracle
    g = np.load(os.path.join(golden_dir, "small_cases.npz"))
    impressions = ["N1-0 N2-1 N3-0", "N2-0 N4-1", "N5-1 N1-0 N6-0 N7-0"]
    history = ["N9 N1 N8", "N8", "N4 N9 N10 N2"]
    sp = split_impressions_and_history(impressions, history)
    assert list(sp["news_list"]) == list(g["split_news"])
    for a, b in (("impression_rev_ind_array", "split_imp"), ("impression_len_list", "split_imp_len"),
                 ("history_rev_ind_array", "split_hist"), ("history_len_list", "split_hist_len")):
        assert np.array_equal(sp[a], g[b]) and sp[a].dtype == np.int32
    assert [list(l) for l in sp["labels"]] == [[0, 1, 0], [0, 1], [1, 0, 0, 0]]
    # random log with missing histories (None / ""), no labels, repeated ids -- against the oracle restatement
    rng = np.random.default_rng(3)
    ids = [f"N{rng.integers(0, 400)}" for _ in range(6000)]
    imps, hists, k = [], [], 0
    for r in range(500):
        c, h = int(rng.integers(1, 9)), int(rng.integers(0, 6))
        imps.append(" ".join(ids[k:k + c]))
        hists.append(None if h == 0 and r % 2 else " ".join(ids[k + c:k + c + h]))
        k += c + h
    want = oracle.split_impressions_and_history(imps, [h if h else "" for h in hists])
    got = split_impressions_and_history(imps, hists)
    assert list(got["news_list"]) == list(want["news_list"]) and len(got["labels"]) == 0
    for key in ("impression_rev_ind_array", "impression_len_list", "history_rev_ind_array", "history_len_list"):
        assert np.array_equal(got[key], want[key])


def test_native_csr_builder_property_vs_oracle_and_live_reference():
    """Random behaviour logs WITH labels (duplicates inside a row, empty / missing histories, one-candidate rows):
    nrb_csr_build == the oracle restatement == the reference itself (when its tree is present)."""
    hypothesis = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st

    from news_recommendation_project_v2_b200.data_utils import split_impressions_and_history
    from oracle import oracle, ref_harness
    ref = ref_harness.load_reference() if ref_harness.reference_available() else None
    news = st.integers(min_value=0, max_value=60).map(lambda i: f"N{i}")
    row = st.tuples(st.lists(st.tuples(news, st.integers(0, 1)), min_size=1, max_size=9),
                    st.one_of(st.none(), st.lists(news, min_size=0, max_size=7)))

    @settings(max_examples=60, deadline=None)
    @given(st.lists(row, min_size=1, max_size=25))
    def check(rows):
        imps = [" ".join(f"{n}-{l}" for n, l in cands) for cands, _ in rows]
        hists = [None if h is None or len(h) == 0 else " ".join(h) for _, h in rows]
        got = split_impressions_and_history(imps, hists)
        want = oracle.split_impressions_and_history(imps, [h if h else "" for h in hists])
        others = [want]
        if ref is not None and any(hists):  # the reference itself raises (np.concatenate of nothing) when NO row has a history
            import pandas as pd
            others.append(ref.data_utils.split_impressions_and_history(
                pd.Series(imps, dtype=object), pd.Series(hists, dtype=object)))
        for w in others:
            assert list(got["news_list"]) == list(w["news_list"])
            for key in ("impression_rev_ind_array", "impression_len_list", "history_rev_ind_array", "history_len_list"):
                assert np.array_equal(got[key], np.asarray(w[key])) and got[key].dtype == np.int32, key
            assert [tuple(int(v) for v in l) for l in got["labels"]] == [tuple(int(v) for v in l) for l in w["labels"]]

    check()


def test_token_store_roundtrip(tmp_path):
    """sqlite token store (reference format) -> packed tokens + CSR offsets."""
    from news_recommendation_project_v2_b200.token_store import read_token_store, write_token_store
    g = torch.Generator().manual_seed(0)
    items = [torch.randn(n, 16, generator=g).half() for n in (3, 1, 7, 2)]
    db = str(tmp_path / "tok.sqlite")
    write_token_store(db, items)
    tokens, off = read_token_store(db, dtype=torch.float32)
    assert off.tolist() == [0, 3, 4, 11, 13] and tokens.shape == (13, 16)
    assert torch.equal(tokens[4:11], items[2].float())
    tokens, off = read_token_store(db, ids=[2, 0, 2], dtype=torch.float32)
    assert off.tolist() == [0, 7, 10, 17] and torch.equal(tokens[7:10], items[0].float())
    with pytest.raises(IndexError):
        read_token_store(db, ids=[9])


def test_packed_token_file_roundtrip(tmp_path):
    """sqlite token store -> packed token file: same tokens (bf16-rounded), same item boundaries, mmap-able, chunk
    bounds cover every item once and respect the token budget."""
    from news_recommendation_project_v2_b200.token_store import (PackedTokenFile, convert_token_store,
                                                                 write_packed_tokens, write_token_store)
    g = torch.Generator().manual_seed(0)
    items = [torch.randn(int(n), 64, generator=g).half() for n in torch.randint(0, 30, (57,), generator=g)]
    db, path = str(tmp_path / "tok.sqlite"), str(tmp_path / "tok.nrbtok")
    write_token_store(db, items)
    n_items, n_tok = convert_token_store(db, path)
    tf = PackedTokenFile(path)
    assert (n_items, n_tok) == (57, sum(t.shape[0] for t in items)) == (tf.n_items, tf.n_tokens) and tf.dim == 64
    assert tf.dtype == torch.bfloat16 and tf.offsets[0] == 0 and tf.offsets[-1] == n_tok
    assert np.array_equal(np.diff(tf.offsets), [t.shape[0] for t in items])
    assert torch.equal(tf.tokens(0, n_tok), torch.cat([t.to(torch.bfloat16) for t in items]))
    bounds = tf.chunk_bounds(64)
    assert bounds[0][0] == 0 and bounds[-1][1] == 57 and all(a[1] == b[0] for a, b in zip(bounds, bounds[1:]))
    assert all(tf.offsets[b] - tf.offsets[a] <= 64 for a, b in bounds)
    # fp32 files and the header check
    write_packed_tokens(str(tmp_path / "f32.nrbtok"), [t.float() for t in items[:5]], 64, torch.float32)
    t32 = PackedTokenFile(str(tmp_path / "f32.nrbtok"))
    assert t32.dtype == torch.float32 and torch.equal(t32.tokens(0, t32.n_tokens), torch.cat(items[:5]).float())
    (tmp_path / "bad.nrbtok").write_bytes(b"x" * 8192)
    with pytest.raises(ValueError):
        PackedTokenFile(str(tmp_path / "bad.nrbtok"))


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the arm the driver times beside ours) prints ONE JSON line with the contract keys;
    under torchrun every rank but 0 exits without work."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--ref-sample", "16"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "impressions_per_sec_scored" and d["unit"] == "impressions/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    # the unmodified reference (oracle/_ref, oracle/build_ref.py) when it is installed, else the oracle port
    from oracle import ref_harness
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_harness.reference_available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
    # argument errors are refused before any work
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"], ["--only-stage-a", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), *bad], capture_output=True, text=True,
                             timeout=600, cwd=root)
        assert out.returncode == 2 and out.stdout == "", out.stderr[-2000:]


def test_bench_dump_outputs_sample(tmp_path):
    """`bench.py --dump-outputs`: whole impressions of a seeded sample, in ascending order, scores and ranks at their
    candidates' positions, float32 / float64 files, within the candidate budget, the same sample on every call."""
    import bench
    g = torch.Generator().manual_seed(1)
    for n_imp in (7, 300_000):
        cnt = torch.randint(2, 301, (n_imp,), generator=g)
        c_off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(cnt, 0)])
        n_c = int(c_off[-1])
        scores = torch.randn(n_c, generator=g)
        ranks = torch.randint(1, 301, (n_c,), generator=g, dtype=torch.int32)
        dumps = []
        for run in range(2):
            d = tmp_path / f"{n_imp}_{run}"
            bench.dump_outputs(str(d), scores, ranks, c_off)
            dumps.append({f.stem: np.load(f) for f in d.glob("*.npy")})
        a = dumps[0]
        assert set(a) == {"scores", "ranks", "impressions", "candidates_per_impression"}
        for k in a:
            assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], dumps[1][k])
        imp = a["impressions"].astype(np.int64)
        assert np.all(np.diff(imp) > 0) and np.array_equal(a["candidates_per_impression"], cnt.numpy()[imp])
        co = c_off.numpy()
        pos = np.concatenate([np.arange(co[i], co[i + 1]) for i in imp])
        assert np.array_equal(a["scores"], scores.numpy()[pos])
        assert np.array_equal(a["ranks"], ranks.numpy()[pos].astype(np.float32))
        if n_imp == 7:
            assert len(imp) == n_imp
        else:
            assert bench.DUMP_MAX_CANDIDATES - 300 < len(pos) <= bench.DUMP_MAX_CANDIDATES
        assert sum(v.nbytes for v in a.values()) <= 64 << 20


def _toy_behaviors():
    import pandas as pd

    beh = pd.DataFrame({
        "ImpressionID": [11, 12, 13, 14],
        # object dtype keeps the missing history as None (the reference's `if hist_row:` relies on that)
        "History": pd.Series(["N3 N1 N3", None, "N7", "N1 N9 N2 N3"], dtype=object),
        "Impressions": pd.Series(["N5-0 N1-1 N6-0", "N2-1 N5-0", "N8-0 N3-1 N1-0 N2-0", "N6-1 N7-0"], dtype=object),
    })
    news = sorted({t.split("-")[0] for r in beh["Impressions"] for t in r.split()} |
                  {t for r in beh["History"].dropna() for t in r.split()})
    rng = np.random.default_rng(5)
    ctx = {
        "behaviors": beh, "news_text_dict": {n: f"text of {n}" for n in news},
        "news_category": {n: int(rng.integers(0, 18)) for n in news},
        "news_subcategory": {n: int(rng.integers(0, 200)) for n in news},
        "news_title_entity": {n: rng.standard_normal(100).astype(np.float32) for n in news},
        "news_abstract_entity": {n: rng.standard_normal(100).astype(np.float32) for n in news},
        "news_dataset": "toy",
    }
    return ctx


def test_transform_data_and_table_components(tmp_path):
    """The components either side of the hot path (components.py:45-114, 178-258): same context keys, dtypes and
    row order as the reference; compared with the reference itself when it is importable here."""
    from news_recommendation_project_v2_b200.components import (LoadEmbeddingComponent, SaveEmbeddingComponent,
                                                                TransformData)
    from news_recommendation_project_v2_b200.config import NewsDataset
    from oracle import oracle

    ctx = _toy_behaviors()
    out = TransformData().transform(dict(ctx))
    want = oracle.split_impressions_and_history(list(ctx["behaviors"]["Impressions"]), list(ctx["behaviors"]["History"]))
    assert list(out["news_list"]) == list(want["news_list"]) and out["news_list"][0] == "N3"  # first appearance
    for k in ("impression_rev_ind_array", "impression_len_list", "history_rev_ind_array", "history_len_list"):
        assert np.array_equal(out[k], want[k]) and out[k].dtype == np.int32
    assert list(out["history_bool"]) == [True, False, True, True]
    assert out["cat_indices"].shape == (len(out["news_list"]), 1) and out["cat_indices"].dtype == torch.int32
    assert out["title_entity_embed"].dtype == torch.float32
    assert torch.equal(out["title_entity_embed"][0], torch.from_numpy(ctx["news_title_entity"]["N3"]))
    assert int(out["subcat_indices"][2, 0]) == ctx["news_subcategory"][out["news_list"][2]]
    for gone in ("behaviors", "news_category", "news_subcategory", "news_title_entity", "news_abstract_entity"):
        assert gone not in out
    assert "news_text_dict" in out and list(out["ImpressionID"]) == [11, 12, 13, 14]
    with pytest.raises(AssertionError):
        TransformData().transform({"behaviors": ctx["behaviors"]})

    if os.path.isdir("/root/reference/src"):
        from oracle import ref_harness
        ref = ref_harness.load_reference()
        ref_out = ref.components.TransformData().transform(dict(ctx))
        assert set(ref_out) == set(out)
        for k, v in ref_out.items():
            if isinstance(v, torch.Tensor):
                assert torch.equal(v, out[k]) and v.dtype == out[k].dtype, k
            elif isinstance(v, np.ndarray) and v.dtype != object:
                assert np.array_equal(v, out[k]) and v.dtype == out[k].dtype, k

    table = torch.randn(len(out["news_list"]), 8)
    ctx2 = {"news_embeddings": table, "query_news_embeddings": table * 2, "news_dataset": NewsDataset.MINDsmall_dev}
    SaveEmbeddingComponent(tmp_path / "emb").transform(ctx2)
    assert (tmp_path / "emb" / "MINDsmall_dev.pt").exists() and (tmp_path / "emb" / "query_MINDsmall_dev.pt").exists()
    back = LoadEmbeddingComponent(tmp_path / "emb").transform({"news_dataset": NewsDataset.MINDsmall_dev})
    assert torch.equal(back["news_embeddings"], table) and torch.equal(back["query_news_embeddings"], table * 2)


def test_integration_stub_matches_the_abi():
    """The reference-side ctypes stub shown in INTEGRATION.md declares the same argument lists as the library."""
    import ctypes as C
    import types

    from news_recommendation_project_v2_b200 import _lib

    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    block = md.split("# news_rec_utils/_nrb200.py")[1].split("```")[0]
    decl = [l for l in block.splitlines() if l.startswith("_lib.") and ("argtypes" in l or "restype" in l)]
    assert len(decl) >= 5
    fake = types.SimpleNamespace(**{n: types.SimpleNamespace() for n in _lib.PROTOTYPES})
    env = {"C": C, "_lib": fake, "P": C.c_void_p, "I64": C.c_int64, "I32": C.c_int}
    exec("\n".join(decl), env)
    for name in ("nrb_final_attention_rows_workspace_bytes", "nrb_final_attention_rows", "nrb_score_rank"):
        want = _lib.PROTOTYPES[name][1]
        got = getattr(fake, name).argtypes
        assert len(got) == len(want), name
        for a, b in zip(got, want):
            assert C.sizeof(a) == C.sizeof(b), (name, a, b)


def test_sass_contains_the_blackwell_instructions():
    """The built sm_100a library really carries tcgen05 / TMEM / TMA code (SASS mnemonics of B200_PROFILING.md):
    UTCHMMA(.2CTA) = tcgen05.mma (CTA pairs), LDTM / STTM = tcgen05.ld / st, UTMALDG / UTMASTG = TMA load / store,
    and 128-bit global loads for the bandwidth-bound kernels."""
    import shutil
    import subprocess

    from news_recommendation_project_v2_b200 import _lib, build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    build.build()
    _lib.load()
    path = os.environ.get("NRB200_LIB") or os.path.join(ROOT, "news_recommendation_project_v2_b200", "libnrb200.so")
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, timeout=600).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTCHMMA.2CTA", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTCBAR", "LDG.E.128"):
        assert mnemonic in sass, f"{mnemonic} missing from the SASS"


def test_balanced_cuts_match_full_array_search():
    """score_host's chunk plan by bisection == np.searchsorted over the full cost array; the tapered plan only adds
    cuts inside the last chunk."""
    from news_recommendation_project_v2_b200.engine import _balanced_cuts
    rng = np.random.default_rng(0)
    for n in (1, 2, 7, 1000, 50_000):
        ho = np.concatenate([[0], np.cumsum(rng.integers(0, 51, n))]).astype(np.int64)
        co = np.concatenate([[0], np.cumsum(rng.integers(1, 55, n))]).astype(np.int64)
        cost = 2 * ho + co
        for nc in (1, 3, 8, 16):
            k = max(1, min(nc, n))
            want = sorted(set([0] + np.searchsorted(cost, cost[-1] * np.arange(1, k) / k).tolist() + [n]))
            got = _balanced_cuts(ho, co, n, k)
            assert got == want
            tapered = _balanced_cuts(ho, co, n, k, taper=True)
            assert set(got) <= set(tapered) and tapered == sorted(tapered) and tapered[0] == 0 and tapered[-1] == n
            assert all(c >= got[-2] for c in set(tapered) - set(got))
