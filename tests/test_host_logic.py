"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/issue_emb_b200.h declares,
it fails loudly without a GPU (no CPU fallback), the bulk driver reproduces the reference's sort / pad / unsort /
OOM-halving logic, and the N>1 sharding + single all-gather works under gloo with world_size 2."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from code_intelligence_b200 import _lib, bulk  # noqa: E402
from oracle import awd_lstm_ref as R  # noqa: E402


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "issue_emb_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(ie_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.PROTOTYPES), (declared ^ set(_lib.PROTOTYPES))
    assert lib.ie_version() >= 100


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from code_intelligence_b200 import IssueEncoder
    from code_intelligence_b200.mlp import MLPHead
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        IssueEncoder(2, 16, 32, 100)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        MLPHead([np.zeros((4, 3), np.float32)], [np.zeros(3, np.float32)])


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "code_intelligence_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{fn} imports the oracle"
                assert "/root/reference" not in src


def _oracle_encoder_fn(enc):
    return lambda ids, lengths: R.encode_padded(enc, ids, lengths)


def test_bulk_loop_matches_reference_driver_restatement():
    enc = R.make_encoder(3, 400, 24, 40, 3, scale=2.0)
    docs = R.synthetic_ids(53, 30, seed=4, vocab_sz=400, min_len=1)
    want = R.encode_bulk(enc, docs, bs=9)                       # restatement of df_to_embedding's loop
    calls = []
    def fn(ids, lengths):
        calls.append(ids.shape)
        return R.encode_padded(enc, ids, lengths)
    got = bulk.encode_sorted_batches(docs, fn, pad_idx=1, out_dim=72, bs=9)
    np.testing.assert_allclose(got, want, atol=1e-6)
    assert got.dtype == np.float32 and got.shape == (53, 72)
    assert calls[0][0] == min(9, 53 // 20 + 1)                  # bs rule: min(bs, N//20 + 1)
    assert all(calls[i][1] <= calls[i + 1][1] for i in range(len(calls) - 1))   # sorted by length


def test_bulk_loop_oom_halving_and_reraise():
    enc = R.make_encoder(3, 400, 24, 40, 2)
    docs = R.synthetic_ids(40, 12, seed=5, vocab_sz=400, min_len=2)
    seen = []
    def flaky(ids, lengths):
        seen.append(ids.shape[0])
        if ids.shape[0] > 2:
            raise RuntimeError("CUDA out of memory (simulated)")
        return R.encode_padded(enc, ids, lengths)
    got = bulk.encode_sorted_batches(docs, flaky, 1, 72, bs=8, min_batches_rule=False)
    np.testing.assert_allclose(got, R.encode_bulk(enc, docs, bs=100), atol=1e-6)
    assert seen[:3] == [8, 4, 2]
    def always(ids, lengths):
        raise RuntimeError("CUDA out of memory (simulated)")
    with pytest.raises(Exception):
        bulk.encode_sorted_batches(docs, always, 1, 72, bs=4)
    assert bulk.encode_sorted_batches([], always, 1, 72).shape == (0, 72)
    with pytest.raises(ValueError):
        bulk.encode_sorted_batches([np.array([], dtype=np.int64)], always, 1, 72)


def test_shard_plan_round_robin():
    lengths = np.array([5, 1, 9, 3, 7, 2, 8])
    order, shards = bulk.shard_plan(lengths, 3)
    assert sorted(np.concatenate(shards).tolist()) == list(range(7))
    assert [lengths[s].tolist() for s in shards] == [[1, 5, 9], [2, 7], [3, 8]]


_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from code_intelligence_b200 import bulk
from oracle import awd_lstm_ref as R
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
enc = R.make_encoder(3, 400, 24, 40, 2)
docs = R.synthetic_ids(37, 20, seed=6, vocab_sz=400, min_len=1)
local = lambda d: bulk.encode_sorted_batches(d, lambda i, l: R.encode_padded(enc, i, l), 1, 72, bs=4, min_batches_rule=False)
out = bulk.encode_bulk_distributed(docs, local)
want = R.encode_bulk(enc, docs, bs=100)
assert out.shape == (37, 72), out.shape
assert np.allclose(out, want, atol=1e-6), np.abs(out - want).max()
# an empty shard on one rank must still work
one = bulk.encode_bulk_distributed(docs[:1], local)
assert np.allclose(one, want[:1], atol=1e-6)
# the per-rank encoder may hand back a tensor (on the GPU: device resident); to_host=False keeps the result a tensor
as_t = bulk.encode_bulk_distributed(docs, lambda d: torch.from_numpy(local(d)), to_host=False)
assert isinstance(as_t, torch.Tensor) and np.array_equal(as_t.numpy(), out)
dist.destroy_process_group()
print("rank", sys.argv[1], "ok")
'''


def test_distributed_bulk_gloo_world2(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "w.py"
    script.write_text(_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_features_dictionary_and_writers(tmp_path):
    """Output contract of get_all_issue_text (py/code_intelligence/embeddings.py:116-118): features[:, :1600]."""
    from code_intelligence_b200 import embeddings as E

    class FakeWrapper:            # stands in for InferenceWrapper: the contract under test is the slicing / writers
        def df_to_embedding(self, df, bs=100):
            return np.arange(len(df) * 2400, dtype=np.float32).reshape(len(df), 2400)

    issues = [dict(title=f"t{i}", body="b", labels=[f"l{i}"], num=i + 1) for i in range(3)]
    d = E.issues_to_features(FakeWrapper(), issues)
    assert d["features"].shape == (3, 1600) and d["labels"] == [["l0"], ["l1"], ["l2"]] and d["nums"] == [1, 2, 3]
    np.testing.assert_array_equal(d["features"][1], np.arange(2400, 2400 + 1600, dtype=np.float32))
    with pytest.raises(ValueError):
        E.issues_to_features(FakeWrapper(), [])
    E.save_features(str(tmp_path / "f.dpkl"), d)
    import dill
    back = dill.load(open(tmp_path / "f.dpkl", "rb"))
    np.testing.assert_array_equal(back["features"], d["features"])
    out = E.save_embeddings(str(tmp_path / "emb"), np.ones((2, 2400)))
    arr = np.load(out) if out.endswith(".npy") else None
    assert arr is None or (arr.dtype == np.dtype("<f4") and arr.shape == (2, 2400))


def test_text_boundary_helpers_cpu_only():
    """process_dict / RuleTokenizer are host-side boundary code (inference.py:92-123, :51-53): markers, fallback text."""
    from code_intelligence_b200.inference import InferenceWrapper, RuleTokenizer, pass_through
    d = InferenceWrapper.process_dict({"title": "Crash in  TFJob", "body": "It FAILS!!!!!"})
    assert d["text"].startswith("xxxfldtitle ") and " xxxfldbody " in d["text"]
    with pytest.raises(AssertionError):
        InferenceWrapper.process_dict({"title": "x"})
    assert InferenceWrapper.process_dict({"title": None, "body": "b"}) == {"text": "xxxUnk"}   # swallowed like the reference
    assert pass_through(3) == 3
    itos = ["xxunk", "xxpad", "xxbos", "xxfld", "xxmaj", "xxup", "xxrep", "xxwrep", "crash", "in", "it", "fails", "!"]
    ids = RuleTokenizer(itos)("Crash in IT fails")
    assert ids.dtype == np.int64 and ids[0] == 2 and list(ids[1:]) == [4, 8, 9, 5, 10, 11]   # xxmaj crash in xxup it fails
    df = __import__("pandas").DataFrame({"title": ["a", "b"], "body": ["c", "d"]})
    assert list(InferenceWrapper.process_df(df)["text"]) == ["xxxfldtitle a xxxfldbody c", "xxxfldtitle b xxxfldbody d"]


def test_spacy_like_tokenizer_documented_cases():
    """Row f-1 (SURVEY.md section 8): the word splitter used when fastai/spaCy are absent.  Expected outputs are the
    behaviours spaCy documents for its English tokenizer (usage docs' "Let's go to N.Y.!" walk-through, the
    contraction / punctuation / unit / hyphen cases of spacy/tests/lang/en) -- unpinned against a live spaCy."""
    from code_intelligence_b200.tokenizer import SpacyLikeTokenizer
    tok = SpacyLikeTokenizer(["xxbos", "xxfld", "xxmaj", "xxup", "xxrep", "xxwrep", "xxunk", "xxpad"])
    cases = {
        "Let's go to N.Y.!": ["Let", "'s", "go", "to", "N.Y.", "!"],
        "I don't think we can't.": ["I", "do", "n't", "think", "we", "ca", "n't", "."],
        "I'm here, it's fine; they're late": ["I", "'m", "here", ",", "it", "'s", "fine", ";", "they", "'re", "late"],
        "Hello, world.": ["Hello", ",", "world", "."],
        "(foo) [bar]": ["(", "foo", ")", "[", "bar", "]"],
        "It costs $10.50, i.e. 10% of 10km...": ["It", "costs", "$", "10.50", ",", "i.e.", "10", "%", "of", "10", "km",
                                                 "..."],
        "a well-known fix": ["a", "well", "-", "known", "fix"],
        "The U.K. and e.g. Mr. Smith": ["The", "U.K.", "and", "e.g.", "Mr.", "Smith"],
        "ok :) <3": ["ok", ":)", "<3"],
        "a\n\nb \n c": ["a", "\n\n", "b", "\n ", "c"],          # whitespace runs other than one space are tokens
        "x=y a:b 1-2 end.Start": ["x", "=", "y", "a", ":", "b", "1", "-", "2", "end", ".", "Start"],
        "see http://example.com/a?b=c now": ["see", "http://example.com/a?b=c", "now"],
        "cannot gonna": ["can", "not", "gon", "na"],
        "xxbos xxmaj hello xxrep 4 !": ["xxbos", "xxmaj", "hello", "xxrep", "4", "!"],
        "C++ and .NET v1.2.3": ["C++", "and", ".NET", "v1.2.3"],
        "": [],
    }
    for text, want in cases.items():
        assert tok(text) == want, (text, tok(text))
    # every character except single separating spaces survives tokenisation, in order
    for text in cases:
        assert "".join(tok(text)).replace(" ", "") == text.replace(" ", "")


def test_rule_tokenizer_reproduces_reference_notebook_tokens(golden_dir):
    """Row f-1 pinned on REFERENCE OUTPUT: the token strings the reference's own pipeline (mdparse + spaCy 2.x + fastai
    rules) printed in Issue_Embeddings/notebooks/04_Inference.ipynb:118-156 -- 41 fragments, 904 tokens (contractions,
    possessives, version numbers, dotted identifiers, '--', '...', hyphenated words, emoji, ctrl+c, xxmaj / xxup / xxrep).
    The notebook shows only the processed side, so each fragment's raw text is its natural detokenisation
    (tests/golden/tokenizer_ref_notebook.json says so; three titles are also printed raw at 02_fastai_DataBunch.ipynb:118-128); fragments with mdparse markers or xxunk were cut out."""
    import json
    from code_intelligence_b200.inference import RuleTokenizer
    fx = json.load(open(os.path.join(golden_dir, "tokenizer_ref_notebook.json"), encoding="utf-8"))
    rt = RuleTokenizer(['xxunk', 'xxpad', 'xxbos', 'xxfld', 'xxmaj', 'xxup', 'xxrep', 'xxwrep'])
    assert len(fx["fragments"]) >= 40
    for f in fx["fragments"]:
        unk = set(f.get("unk", []))          # words the reference's 60 000-word vocabulary did not hold
        got = ["xxunk" if t in unk else t for t in rt.tokens(f["raw"])]
        assert got == f["tokens"].split(" "), f["raw"]


def test_rule_tokenizer_process_text_pipeline():
    """fastai Tokenizer.process_text restated: pre-rules -> splitter -> post-rules -> vocab lookup."""
    from code_intelligence_b200.inference import RuleTokenizer
    itos = ['xxunk', 'xxpad', 'xxbos', 'xxfld', 'xxmaj', 'xxup', 'xxrep', 'xxwrep', 'wow', '!', 'this', 'is', 'cool',
            '5', "n't", 'does', 'work', '#', '12', '/']
    rt = RuleTokenizer(itos)
    toks = rt.tokens("WOW!!!!! This is is is is is cool")
    assert toks == ['xxup', 'wow', 'xxrep', '5', '!', 'xxmaj', 'this', 'xxwrep', '5', 'is', 'cool'], toks
    ids = rt("Doesn't work #12 a/b")
    want = ['xxbos', 'xxmaj', 'does', "n't", 'work', '#', '12', 'xxunk', '/', 'xxunk']
    assert [itos[i] for i in ids] == want, [itos[i] for i in ids]
    assert ids.dtype == np.int64 and ids[0] == 2


def test_bench_clock_sampler_summary():
    """bench.py's `clocks` key: the median SM clock / power over the samples taken under load, throttle reasons."""
    import bench
    idle = ["0", "1965", "1965", "180.2", "x", "Not Active", "Not Active", "Not Active", "Not Active"]
    busy = ["0", "1400", "1965", "990.1", "x", "Not Active", "Not Active", "Not Active", "Active"]
    s = bench.ClockSampler.summarise([idle] * 5 + [busy] * 7 + [["garbage"]])
    assert s["sm_mhz"] == 1400.0 and s["sm_max_mhz"] == 1965.0 and s["reasons"] == ["sw_power_cap"]
    assert s["samples"] == 12 and s["samples_under_load"] == 7 and s["power_w"] == 990.1
    assert bench.ClockSampler.summarise([])["sm_mhz"] is None


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: float32 .npy per name, a row sample that is the same on every run, a size cap."""
    import bench
    a = np.arange(5000 * 3, dtype=np.float64).reshape(5000, 3)
    s = bench.sample_rows(a, 1024)
    assert s.shape == (1024, 3) and np.array_equal(s, bench.sample_rows(a, 1024))
    assert (np.diff(s[:, 0]) > 0).all() and np.isin(s[:, 0], a[:, 0]).all()
    small = bench.sample_rows(a[:10], 1024)
    assert np.array_equal(small, a[:10]) and not np.shares_memory(small, a)
    bench.dump_outputs(str(tmp_path / "d"), {"embeddings": a[:4], "e2e_embeddings_sample": s})
    back = np.load(tmp_path / "d" / "embeddings.npy")
    assert back.dtype == np.float32 and np.array_equal(back, a[:4].astype(np.float32))
    assert sorted(os.listdir(tmp_path / "d")) == ["e2e_embeddings_sample.npy", "embeddings.npy"]
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros((bench.DUMP_MAX_BYTES // 4 + 1,), np.float32)})


def _rot_schedule_model(T, ng, tiles, P, mma, lat, slots=2, pre=0.0):
    """Event model of csrc/lstm_layer.cu's schedule: item n = t*C + g*tiles + j (C = ng*tiles) runs on CTA pair n % P, pairs
    walk their items in increasing n; an item's MMAs start when the pair is free, every item of (t-1, g) has been
    published (its MMA end + lat) and the pair's item `slots` positions back has left its TMEM slot (MMA end + lat).
    `pre`: MMA time of the item that does NOT depend on (t-1, g) -- the fused input projection of the last layer (FUSE):
    it starts as soon as the pair and the TMEM slot are free, only the remaining `mma` waits for the counter.
    Returns (makespan, items seen, True if every dependency had a smaller index)."""
    C, total = ng * tiles, T * ng * tiles
    end, pub, cnt, tile_pub, pair_free = {}, {}, {}, {}, [0.0] * P
    seen, ordered = set(), True
    for n in range(total):                      # ascending n is a valid evaluation order iff deps have smaller indices
        p, k = n % P, n // P
        t, c = divmod(n, C)
        g, j = divmod(c, tiles)
        seen.add((t, g, j))
        start = pair_free[p]
        if k >= slots:
            start = max(start, end[n - slots * P] + lat)
        start += pre                            # the dependency-free part runs first
        if t > 0:
            if (t - 1, g) not in pub:           # some tile of (t-1, g) has an index >= n: the order argument would break
                ordered = False
                break
            start = max(start, pub[(t - 1, g)])
        end[n] = pair_free[p] = start + mma
        tile_pub[(t, g)] = max(tile_pub.get((t, g), 0.0), end[n] + lat)
        cnt[(t, g)] = cnt.get((t, g), 0) + 1
        if cnt[(t, g)] == tiles:
            pub[(t, g)] = tile_pub[(t, g)]
    return (max(end.values()) + lat if end else 0.0), len(seen), ordered


def test_rotating_schedule_model():
    """Design claims of DESIGN.md section 4 / csrc/lstm_layer.cu, checked on a timing model: every (t, batch, tile) item is
    dealt exactly once, an item only waits for smaller indices (=> no wait cycle for ANY pair count), and with five
    batches at H = 2400 (C = 190 >= 2*74 + 38) the pairs issue back to back (within 2 % of 38*mma/74 per batch-step)
    although each item's inputs take `lat` to become visible, while three batches leave that latency exposed."""
    for (T, ng, tiles, P) in ((5, 1, 1, 74), (7, 3, 38, 74), (4, 5, 38, 74), (6, 5, 13, 74), (9, 2, 4, 3), (3, 5, 38, 1)):
        span, n_items, ordered = _rot_schedule_model(T, ng, tiles, P, mma=1.0, lat=0.7)
        assert ordered and n_items == T * ng * tiles and span > 0
    mma, lat, T = 13.8, 8.0, 48
    ideal = 38 * mma / 74
    per_step = {ng: _rot_schedule_model(T, ng, 38, 74, mma, lat)[0] / T / ng for ng in (3, 5)}
    assert per_step[5] <= 1.02 * ideal, per_step
    assert per_step[3] >= 1.15 * ideal, per_step          # 114 items per timestep: the dependency latency shows


def test_fused_last_layer_hides_its_step_chain_in_the_model():
    """Why the last layer's input projection rides its recurrent K loop (DESIGN.md section 4, csrc/lstm_layer.cu FUSE): with
    13 tiles x 5 batches = 65 items per timestep on 74 pairs every pair has at most one item per timestep, so the hoisted
    form is bound by the step chain (MMA + visibility latency per timestep) and the projection GEMM comes on top; with the
    38 dependency-free k-blocks in front of the 13 recurrent ones the chain hides behind the item itself and the layer
    runs at the rate of its MMA stream (65 / 74 of a pair per timestep).  Times in units of one k-block."""
    T, ng, tiles, P = 64, 5, 13, 74
    rec, pre, lat = 13.0, 38.0, 22.0          # k-blocks; visibility latency ~ epilogue + publish + counter + first tile
    hoisted = _rot_schedule_model(T, ng, tiles, P, mma=rec, lat=lat)[0] / T
    fused, n_items, ordered = _rot_schedule_model(T, ng, tiles, P, mma=rec, lat=lat, pre=pre)
    fused /= T
    assert ordered and n_items == T * ng * tiles
    assert hoisted >= 0.95 * (rec + lat)                         # chain-bound: one MMA phase + one latency per timestep
    gemm_equiv = pre * ng * tiles / P                            # the hoisted projection at full rate, per timestep
    stream = (pre + rec) * ng * tiles / P                        # all 51 k-blocks of the 65 items on 74 pairs
    assert fused <= 1.12 * stream, (fused, stream)               # MMA-stream-bound, chain hidden
    assert fused <= 0.80 * (hoisted + gemm_equiv), (fused, hoisted, gemm_equiv)


def test_bulk_loop_coalesces_reference_batches():
    """`coalesce=True` (the default of IssueEncoder.encode_id_list): the reference's bs (default 100) no longer decides
    the device batch; consecutive sorted batches are merged into calls of max_bs rows, OOM halving still applies, and
    the result equals the un-merged loop because a row's output is independent of its batch mates."""
    enc = R.make_encoder(3, 400, 24, 40, 2)
    docs = R.synthetic_ids(230, 20, seed=6, vocab_sz=400, min_len=1)
    calls = []
    def fn(ids, lengths):
        calls.append(ids.shape)
        if ids.shape[0] > 96:
            raise RuntimeError("CUDA out of memory (simulated)")
        return R.encode_padded(enc, ids, lengths)
    want = bulk.encode_sorted_batches(docs, lambda i, l: R.encode_padded(enc, i, l), 1, 72, bs=10)
    got = bulk.encode_sorted_batches(docs, fn, 1, 72, bs=10, max_bs=768, coalesce=True)
    np.testing.assert_allclose(got, want, atol=1e-6)
    assert [c[0] for c in calls[:3]] == [230, 115, 57]            # everything in one call, then halving until it fits
    assert sum(c[0] for c in calls if c[0] <= 96) == 230
    assert all(calls[i][1] <= calls[i + 1][1] for i in range(2, len(calls) - 1))


def test_c_abi_from_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: include/issue_emb_b200.h must compile as C99 (-pedantic -Werror), every declared
    entry point must link from libissue_emb_b200.so, and without a GPU creation must fail with IE_ERR_CUDA and the
    "no CPU fallback" message (tests/c_abi/abi_check.c)."""
    import subprocess
    from code_intelligence_b200 import _lib
    _lib.load()                                            # builds the library if needed
    libdir = os.path.dirname(_lib.LIB_PATH)
    exe = str(tmp_path / "abi_check")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "c_abi", "abi_check.c"), "-o", exe, "-L", libdir,
                    "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "version=200 symbols=20" in r.stdout, r.stdout


def test_spacy_like_tokenizer_never_loses_characters():
    """Property (hypothesis): for arbitrary text the splitter terminates and its tokens, concatenated, are the input with
    only single separating spaces removed -- no character is dropped, duplicated or reordered."""
    from hypothesis import given, settings, strategies as st
    from code_intelligence_b200.tokenizer import SpacyLikeTokenizer
    tok = SpacyLikeTokenizer(["xxbos", "xxmaj", "xxup"])
    alphabet = st.sampled_from(list("abcXYZ019 .,;:!?'\"()[]{}<>-_/#@$%&*+=~`\n\t’“”…—") + ["n't", "'s", "...", "xxmaj", "e.g.", ":)"])

    @settings(max_examples=300, deadline=None, derandomize=True)
    @given(st.lists(alphabet, max_size=40).map("".join))
    def check(text):
        toks = tok(text)
        assert all(t != "" for t in toks)
        assert "".join(toks).replace(" ", "") == text.replace(" ", "")

    check()


def _driver_fixture(golden_dir):
    z = np.load(os.path.join(golden_dir, "reference_driver.npz"))
    cases = {}
    for tag in ("a", "b", "c"):
        lens = z[f"{tag}_lengths"].astype(np.int64)
        offs = np.concatenate([[0], np.cumsum(lens)])
        docs = [z[f"{tag}_ids"][offs[i]:offs[i + 1]].astype(np.int64) for i in range(len(lens))]
        cases[tag] = dict(docs=docs, bs=int(z[f"{tag}_bs"]), fail_above=int(z[f"{tag}_fail_above"]), expected=z[f"{tag}_expected"])
    return z, cases


def test_bulk_loop_and_pooling_vs_the_reference_driver(golden_dir):
    """Rows a6 / a8 / a9 pinned on the REFERENCE'S OWN CODE: tests/golden/reference_driver.npz holds what
    py/code_intelligence/inference.py's df_to_embedding (:138-229), batch_seq_pool (:232-263) and get_pooled_features
    (:74-92) returned when executed in the build container around the CPU oracle's nn.LSTM stack (generator:
    make_golden.py driver -- only the absent third-party imports and the text -> ids step are stand-ins).  This repo's
    host-side bulk loop, pooling and single-issue path around the same oracle must reproduce those arrays; the OOM
    case (forward calls above 5 rows raise RuntimeError) exercises both halving loops."""
    from code_intelligence_b200 import bulk
    from code_intelligence_b200.inference import InferenceWrapper
    z, cases = _driver_fixture(golden_dir)
    n_layers, emb_sz, n_hid, vocab = [int(v) for v in z["cfg"]]
    ref = R.make_encoder(int(z["seed"]), vocab, emb_sz, n_hid, n_layers, scale=float(z["scale"]))
    for tag, c in cases.items():
        def enc(ids, lengths, c=c):
            if c["fail_above"] >= 0 and ids.shape[0] > c["fail_above"]:
                raise RuntimeError("CUDA out of memory (stub)")
            return R.encode_padded(ref, ids, lengths)
        got = bulk.encode_sorted_batches(c["docs"], enc, pad_idx=1, out_dim=3 * emb_sz, bs=c["bs"])
        np.testing.assert_allclose(got, c["expected"], rtol=0, atol=2e-6, err_msg=tag)
        if c["fail_above"] < 0:      # the oracle's own restatement of the driver (what the GPU tests are checked against)
            np.testing.assert_allclose(R.encode_bulk(ref, c["docs"], bs=c["bs"]), c["expected"], rtol=0, atol=2e-6)
            # ... and the flask_app copy of the driver (Issue_Embeddings/flask_app/inference.py:136-212), also executed
            np.testing.assert_allclose(got, z[f"{tag}_expected_flask_app"], rtol=0, atol=2e-6)
    # pooling and the single-issue path on their own
    np.testing.assert_array_equal(InferenceWrapper.batch_seq_pool(z["pool_seq"], z["pool_lengths"]), z["pool_expected"])
    np.testing.assert_array_equal(R.batch_seq_pool(z["pool_seq"], z["pool_lengths"]), z["pool_expected"])
    one = z["single_ids"].astype(np.int64)
    np.testing.assert_allclose(R.encode_single(ref, one), z["single_expected"], rtol=0, atol=2e-6)


def _check_thresholds_fixture(fn, golden_dir):
    z = np.load(os.path.join(golden_dir, "thresholds_ref.npz"))
    for tag in ("a", "b", "c"):
        thr, prec, rec = fn(z[f"{tag}_scores"], z[f"{tag}_truth"], float(z[f"{tag}_p_thr"]), float(z[f"{tag}_r_thr"]))
        want = z[f"{tag}_thresholds"]
        assert [t is None for t in thr] == list(np.isnan(want)), tag
        np.testing.assert_array_equal(np.array([np.nan if t is None else np.float32(t) for t in thr], dtype=np.float64),
                                      want)                       # thresholds are score values (f32): exact
        np.testing.assert_array_equal(np.array(prec), z[f"{tag}_precisions"])
        np.testing.assert_array_equal(np.array(rec), z[f"{tag}_recalls"])
    assert np.isnan(z["a_thresholds"]).any() and not np.isnan(z["a_thresholds"]).all()


def test_threshold_search_host_restatement_vs_reference_fixture(golden_dir):
    """Row f-4 pinned on the reference: tests/golden/thresholds_ref.npz holds thresholds / precisions / recalls computed
    by the reference's own MLPWrapper.find_probability_thresholds loop (py/label_microservice/mlp.py:65-98; generator:
    make_golden.py thresholds) on preset scores -- ties, a label without positives, excluded labels.  The host restatement
    (the checker of the device kernel in tests/test_gpu_parity.py) must reproduce them exactly."""
    from code_intelligence_b200.mlp import pr_thresholds_host
    _check_thresholds_fixture(pr_thresholds_host, golden_dir)


def test_filter_predictions_reference_case():
    """The reference's own test of the label filter (py/label_microservice/repo_specific_model_test.py:10-33): mocked
    probabilities [[.2, .9]] with thresholds .5 / .5 give {"label2": .9}; a falsy threshold removes the label."""
    from code_intelligence_b200.mlp import filter_predictions
    assert filter_predictions(["label1", "label2"], [.2, .9], {"label1": .5, "label2": .5}) == {"label2": .9}
    assert filter_predictions(["a", "b", "c"], [.9, .9, .4], {"a": None, "b": 0, "c": .3}) == {"c": .4}
    assert filter_predictions([], [], {}) == {}
