"""CPU tests of the host-side mirror: C-ABI exports, mask encoding, prompt layout, DP sharding (gloo)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

from oracle import janus_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_and_exports_every_declared_symbol():
    from plangen_b200 import _lib, build
    lib = build.build()
    cdll = ctypes.CDLL(lib)
    header = open(os.path.join(ROOT, "include", "plangen_b200.h")).read()
    declared = set(re.findall(r"\b(pg_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(cdll, name), f"{name} declared in include/plangen_b200.h but not exported"
    assert declared == set(_lib.EXPORTS), "ctypes table and header disagree"
    m = re.search(r"#define PG_ABI_VERSION (\d+)", header)
    assert cdll.pg_abi_version() == int(m.group(1))


def test_prefill_row_grouping_host_logic():
    """pg_host_group_rows (host half of the prefill's repeated-row shortcut): the first row with the same left padding and
    content hash is proposed as the source; equal hashes with different padding, or equal padding with different hashes, are
    not grouped; the first member of a group points at itself."""
    import numpy as np
    from plangen_b200 import _lib
    lib = _lib.load()
    start = np.array([5, 40, 5, 40, 7, 40, 5, 41], dtype=np.int32)
    h = np.array([11, 99, 11, 99, 11, 98, 12, 99], dtype=np.uint64)
    out = np.full(8, -1, dtype=np.int32)
    n = lib.pg_host_group_rows(start.ctypes.data, h.ctypes.data, 8, out.ctypes.data)
    assert n == 2 and out.tolist() == [0, 1, 0, 1, 4, 5, 6, 7]
    # parallel_size = 2 layout (rows repeat 2B later) and the shared negative prompt (odd rows)
    start = np.array([0, 9, 3, 9, 0, 9, 3, 9], dtype=np.int32)
    h = np.array([1, 7, 2, 7, 1, 7, 2, 7], dtype=np.uint64)
    n = lib.pg_host_group_rows(start.ctypes.data, h.ctypes.data, 8, out.ctypes.data)
    assert n == 5 and out.tolist() == [0, 1, 2, 1, 0, 1, 2, 1]
    assert lib.pg_host_group_rows(start.ctypes.data, h.ctypes.data, 0, out.ctypes.data) == 0
    assert lib.pg_host_group_rows(None, h.ctypes.data, 4, out.ctypes.data) < 0


def test_engine_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from plangen_b200.config import Dims
    from plangen_b200.engine import FastJanus
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        FastJanus({}, Dims.from_any(O.TINY))
    # and the C-ABI itself refuses too
    from plangen_b200 import _lib
    lib = _lib.load()
    pd = _lib.PgDims(); pd.head_dim = 128; pd.vq_nres = 1
    h = ctypes.c_void_p()
    assert lib.pg_engine_create(ctypes.byref(pd), 0, ctypes.byref(h)) != 0
    assert lib.pg_last_error()


def test_kv_start_from_mask_contract():
    from plangen_b200.engine import kv_start_from_mask
    m = torch.tensor([[0, 0, 1, 1, 1, 1, 1], [1, 1, 1, 1, 1, 1, 1], [0, 0, 0, 0, 1, 1, 1]], dtype=torch.int32)
    assert kv_start_from_mask(m, 4).tolist() == [2, 0, 4]          # row 2: empty prompt
    with pytest.raises(ValueError):
        kv_start_from_mask(torch.tensor([[1, 0, 1, 1, 1]]), 3)      # hole: not LEFT padded
    with pytest.raises(ValueError):
        kv_start_from_mask(torch.tensor([[0, 1, 1, 1, 0]]), 3)      # image part must be all ones


def test_collate_mirror_matches_oracle():
    from plangen_b200 import synthetic
    from plangen_b200.config import Dims
    d = Dims.from_any(O.SMALL)
    cond, neg = synthetic.layoutsam_prompts(d, 5, seed=3, lo=9, hi=40, neg_len=11)
    ids, mask = synthetic.collate_cfg_batch(cond, neg, d.pad_id, d.n_img_tokens)
    ids2, mask2 = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    assert torch.equal(ids, ids2) and torch.equal(mask, mask2)
    assert all(d.pad_id not in c for c in cond)
    # ragged + empty rows
    ids, mask = synthetic.collate_cfg_batch([[1, 2, 3], []], [[4], [5, 6]], d.pad_id, 4)
    assert ids.tolist() == [[1, 2, 3], [d.pad_id, d.pad_id, 4], [d.pad_id] * 3, [d.pad_id, 5, 6]]
    assert mask[2].tolist() == [0, 0, 0, 1, 1, 1, 1]


def test_synthetic_state_dict_names_match_oracle_specs():
    from plangen_b200 import synthetic
    from plangen_b200.config import Dims
    for d in (O.TINY, O.SMALL):
        a = [(n, s) for n, s, _ in synthetic.state_dict_names(Dims.from_any(d))]
        b = [(n, s) for n, s, _ in O.tensor_specs(d)]
        assert sorted(a) == sorted(b)
        a = [(n, s) for n, s, _ in synthetic.state_dict_names(Dims.from_any(d), with_vq_encoder=True)]
        b = [(n, s) for n, s, _ in O.tensor_specs(d, with_vq_encoder=True)]
        assert sorted(a) == sorted(b)


def test_weight_bytes_per_step_matches_baseline_md():
    """BASELINE.md §4: 1 275 207 680 weight elements per decode step at 1.3B incl. gen_aligner (4 214 784),
    which the engine replaces by a table gather."""
    from plangen_b200.config import JANUS_1P3B as d
    HD = d.H * d.head_dim
    el = d.L * (3 * HD * d.D + d.D * HD + 3 * d.D * d.F + 2 * d.D) + d.D + (d.D * d.img_embed + d.img_embed + d.img_vocab * d.img_embed + d.img_vocab)
    assert el == 1275207680 - 4214784


def test_shard_batches_round_robin():
    from plangen_b200 import dp
    per_rank = [dp.shard_batches(10, r, 4) for r in range(4)]
    assert per_rank == [[0, 4, 8], [1, 5, 9], [2, 6], [3, 7]]
    assert dp.interleave_results(per_rank, 4) == list(range(10))


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from plangen_b200 import dp
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
mine = dp.shard_batches(5, rank, world)
local = torch.full((2, 3, 4, 4), rank, dtype=torch.uint8)
allimg = dp.gather_images(local, world)
assert allimg.shape == (2 * world, 3, 4, 4) and allimg[2 * rank].eq(rank).all() and allimg[2 * (1 - rank)].eq(1 - rank).all()
# unequal shares (5 batches over 2 ranks): rank 0 holds 3 images, rank 1 holds 2; nobody hangs, order is rank-major
uneven = dp.gather_images(torch.full((len(mine), 3, 4, 4), 10 + rank, dtype=torch.uint8), world)
assert uneven.shape == (5, 3, 4, 4) and uneven[:3].eq(10).all() and uneven[3:].eq(11).all()
only0 = dp.gather_images(torch.full((1 if rank == 0 else 0, 3, 4, 4), 7, dtype=torch.uint8), world)
assert only0.shape == (1, 3, 4, 4) and only0.eq(7).all()
t = dp.max_over_ranks(1.0 + rank, torch.device("cpu"))
assert t == float(world)
sys.stdout.write("rank %d batches %s\n" % (rank, mine)); sys.stdout.flush()
dist.destroy_process_group()
"""


def test_dp_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29517", str(script), ROOT],
                       capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rank 0 batches [0, 2, 4]" in r.stdout and "rank 1 batches [1, 3]" in r.stdout, r.stdout


# ------------------------------------------------------------------ host prompt pipeline (SURVEY §8f rank 4)
class _CharTok:
    """Toy tokenizer for host-logic tests: one id per character (no vocabulary files offline)."""

    def encode(self, s):
        return [ord(c) % 900 + 10 for c in s]

    def decode(self, ids):
        return "".join(chr((int(t) - 10) % 900) for t in ids)


def test_sft_prompt_matches_reference_conversation_template():
    """`want` holds the prompts the reference's own `get_conv_template("deepseek")` (Janus conversation.py) builds for
    these conversations with an empty system message (its stripped `get_prompt()`)."""
    from plangen_b200 import prompts as PR
    convs = [
        [{"role": PR.USER, "content": "a yellow car in front of the tree"}, {"role": PR.ASSISTANT, "content": ""}],
        [{"role": PR.USER, "content": "  two cats "}, {"role": PR.ASSISTANT, "content": "<grounding><ref>cat</ref><box>[1, 2, 3, 4]</box></grounding>"}],
        [{"role": PR.USER, "content": "x"}, {"role": PR.ASSISTANT, "content": "y"}, {"role": PR.USER, "content": "z"}, {"role": PR.ASSISTANT, "content": ""}],
    ]
    want = [
        "<|User|>: a yellow car in front of the tree\n\n<|Assistant|>:",
        "<|User|>: two cats\n\n<|Assistant|>: <grounding><ref>cat</ref><box>[1, 2, 3, 4]</box></grounding><｜end▁of▁sentence｜>",
        "<|User|>: x\n\n<|Assistant|>: y<｜end▁of▁sentence｜><|User|>: z\n\n<|Assistant|>:",
    ]
    assert [PR.sft_prompt(c) for c in convs] == want
    assert PR.sft_prompt(convs[0], system_prompt="be brief") == "be brief\n\n" + want[0]


def test_prompt_pipeline_wraps_pads_and_collates_like_the_reference():
    from plangen_b200 import prompts as PR
    from oracle import janus_oracle as O
    tok = _CharTok()
    pp = PR.PromptPipeline(tok, pad_id=5, image_token_num=16, neg_prompt="bad")
    p_t2i, ids_t2i = pp.wrap_t2i_prompt("a dog")
    assert p_t2i == "<|User|>: a dog\n\n<|Assistant|>:<begin_of_image>" and ids_t2i.tolist() == tok.encode(p_t2i)
    p_uni, ids_uni = pp.wrap_uni_prompt("a dog", "<grounding>G</grounding>")
    assert p_uni.endswith("<grounding>G</grounding><｜end▁of▁sentence｜><begin_of_image>")
    p_s1, ids_s1 = pp.wrap_uni_prompt("a dog", "<grounding>", in_stage1=True)
    assert p_s1 == "<|User|>: a dog\n\n<|Assistant|>: <grounding><｜end▁of▁sentence｜>" and ids_s1.tolist() == tok.encode(p_s1)[:-1]
    caps, grs = ["a dog", "two red birds on a wire"], ["<grounding>A</grounding>", "<grounding>BB</grounding>"]
    uni_ids, uni_mask = pp.uni_batch(caps, grs)
    assert uni_mask.shape[1] == uni_ids.shape[1] + 16 and bool((uni_mask[:, -16:] == 1).all())
    assert bool((uni_ids[0, :(uni_mask[0, :uni_ids.shape[1]] == 0).sum()] == 5).all())          # LEFT padding with pad_id
    ids, mask = pp.t2i_infer_collate_batch(uni_ids, uni_mask)
    cond = [pp.wrap_uni_prompt(c, g)[1].tolist() for c, g in zip(caps, grs)]
    neg = [pp.wrap_uni_prompt("bad", "")[1].tolist()] * 2
    want_ids, want_mask = O.t2i_infer_collate_batch(cond, neg, 5, 16)
    assert ids.dtype == torch.int32 and torch.equal(ids, want_ids) and torch.equal(mask, want_mask)
    # per-sample negatives longer than every cond prompt: the cond side is padded on the left (plangen_base.py:656-662)
    long_neg = (["x" * 80, "y" * 90], ["<grounding></grounding>"] * 2)
    ids2, mask2 = pp.t2i_infer_collate_batch(uni_ids, uni_mask, neg=long_neg)
    negs = [pp.wrap_uni_prompt(c, g)[1].tolist() for c, g in zip(*long_neg)]
    w2_ids, w2_mask = O.t2i_infer_collate_batch(cond, negs, 5, 16)
    assert torch.equal(ids2, w2_ids) and torch.equal(mask2, w2_mask)
    # stage-1 output parsing (plangen_base.py:296-306)
    rows = [tok.encode("<ref>cat</ref></grounding> trailing"), tok.encode("no closing tag")]
    assert pp.decode_plan_text_batch(rows) == ["<grounding><ref>cat</ref></grounding>", "<grounding></grounding>"]


def test_bench_reference_arm_prints_the_contract_line(capsys):
    """`bench.py --impl reference` (the reference's CPU path = oracle port on the host cores): one JSON line with the
    keys the driver reads, on the B200 arm's metric / unit, `impl: reference`, a cpu_baseline describing the run and an
    e2e block with zero copy bytes.  Run on the tiny preset so it takes seconds."""
    import argparse
    import json
    import bench
    args = argparse.Namespace(model="tiny", gpus=1, steps=2, warmup=1, impl="reference")
    os.environ.pop("RANK", None)
    bench.run_reference_arm(args)
    lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["vs_baseline"] is None
    # nothing is extrapolated: one full image per step, the line's time is the wall time of the images that were run
    assert d["steps"] == 2 and d["timed"]["images"] == 2 and d["timed"]["decode_steps"] == 2 * (O.TINY.n_img_tokens - 1)
    assert abs(d["ms_per_step"] * d["steps"] - 1e3 * d["timed"]["wall_s"]) < 1e-6 * d["timed"]["wall_s"] * 1e3 + 1e-9
    assert abs(d["value"] * d["timed"]["wall_s"] - d["steps"]) < 1e-9
    assert d["cpu_baseline_b16"]["images_per_s_estimate"] > 0
    # ranks other than 0 do no work and print nothing
    os.environ["RANK"] = "1"
    try:
        bench.run_reference_arm(args)
        assert capsys.readouterr().out.strip() == ""
    finally:
        os.environ.pop("RANK", None)


def test_bench_dump_outputs_float32_within_budget(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: the step's images and tokens and their batch rows as float32 .npy; a batch over the
    byte budget is cut to the same seeded sample of whole images on every call; a later dump into the same directory
    leaves no file of the earlier one behind."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(0)
    images = torch.randint(0, 256, (6, 3, 8, 8), generator=g, dtype=torch.uint8)
    tokens = torch.randint(0, 16384, (6, 10), generator=g, dtype=torch.int32)

    def load(d):
        assert sorted(os.listdir(d)) == ["images.npy", "rows.npy", "tokens.npy"]
        got = {n: np.load(d / (n + ".npy")) for n in ("images", "tokens", "rows")}
        assert all(a.dtype == np.float32 for a in got.values())
        return got

    budget = bench.DUMP_BYTES
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 4 * (3 * 8 * 8 + 10 + 1))         # room for 4 of the 6 images
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), images, tokens)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    r = a["rows"].astype(np.int64)
    assert len(r) == 4 and np.all(np.diff(r) > 0) and np.array_equal(a["rows"], b["rows"])
    assert np.array_equal(a["images"], images.numpy()[r]) and np.array_equal(a["tokens"], tokens.numpy()[r])
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES + 3 * 128   # + .npy headers
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    bench.dump_outputs(str(tmp_path / "a"), images, tokens)                          # the whole batch fits
    a = load(tmp_path / "a")
    assert np.array_equal(a["rows"], np.arange(6)) and np.array_equal(a["images"], images.numpy())
    assert np.array_equal(a["tokens"], tokens.numpy())


# ------------------------------------------------------------------ teacher-forcing gate (ADVICE r1, plangen_base.py:528,593)
def test_teacher_inputs_validation_and_padding():
    """`_teacher_inputs` mirrors the reference's override loop: exactly `len(edit_region)` rows are overridden, rows of
    further parallel copies are sampled freely (edit_region = 1), malformed shapes are rejected."""
    import types
    import torch
    from plangen_b200.engine import FastJanus
    stub = types.SimpleNamespace(device=torch.device("cpu"))
    f = FastJanus._teacher_inputs
    er = torch.zeros(2, 6, dtype=torch.int64)
    gt = torch.arange(12).reshape(2, 6)
    e, g = f(stub, {"edit_region": er}, gt, 2, 6)
    assert e.dtype == torch.int32 and e.shape == (2, 6) and g.tolist() == gt.tolist()
    e, g = f(stub, {"edit_region": er}, gt, 4, 6)                     # parallel_size = 2: rows 2, 3 are free
    assert e.shape == (4, 6) and e[:2].eq(0).all() and e[2:].eq(1).all() and g[:2].tolist() == gt.tolist()
    e, g = f(stub, {"edit_region": er}, gt, 2, 4)                     # fewer steps than columns: leading columns
    assert e.shape == (2, 4) and g.tolist() == gt[:, :4].tolist()
    for bad in (lambda: f(stub, None, gt, 2, 6), lambda: f(stub, {"edit_region": er}, None, 2, 6),
                lambda: f(stub, {"edit_region": er}, gt[:1], 2, 6), lambda: f(stub, {"edit_region": er}, gt, 1, 6),
                lambda: f(stub, {"edit_region": er}, gt, 2, 7)):
        with pytest.raises(ValueError):
            bad()


def test_kv_start_from_mask_contract():
    import torch
    from plangen_b200.engine import kv_start_from_mask
    m = torch.tensor([[0, 0, 1, 1, 1, 1], [1, 1, 1, 1, 1, 1], [0, 0, 0, 0, 1, 1]])
    assert kv_start_from_mask(m, 4).tolist() == [2, 0, 4]
    with pytest.raises(ValueError):
        kv_start_from_mask(torch.tensor([[1, 0, 1, 1, 1, 1]]), 4)
    with pytest.raises(ValueError):
        kv_start_from_mask(torch.tensor([[0, 1, 1, 1, 0, 1]]), 4)


# ------------------------------------------------------------------ mmu host pipeline + PNG writer (SURVEY 8f rank 4 remainder)
def test_mmu_batchify_layout_matches_the_reference_processor_contract():
    """plangen_base.py:807-841 / processing_vlm.py:215-258, :361-423: each `<image_placeholder>` becomes boi + n image slots + eoi,
    rows are LEFT padded, images_seq_mask marks exactly the image slots and selects as many positions as images_emb_mask."""
    import torch
    from plangen_b200.prompts import PromptPipeline, MMU_QUESTION, IMAGE_PLACEHOLDER

    class Tok(_CharTok):
        def encode(self, s):
            out = []
            for part in s.split(IMAGE_PLACEHOLDER):
                out += super().encode(part) + [5000]
            return out[:-1]

    n_img = 6
    pp = PromptPipeline(Tok(), pad_id=3, image_token_num=n_img, image_id=5000, image_start_id=5001, image_end_id=5002)
    one = pp.mmu_process_one(torch.zeros(1, 3, 8, 8), answer="")
    ids = one["input_ids"].tolist()
    k = ids.index(5001)
    assert ids[k:k + n_img + 2] == [5001] + [5000] * n_img + [5002] and ids.count(5000) == n_img
    assert one["sft_format"].startswith("<|User|>: " + IMAGE_PLACEHOLDER + "\n" + MMU_QUESTION) and one["sft_format"].endswith("<|Assistant|>:")
    imgs = torch.arange(2 * 3 * 8 * 8, dtype=torch.float32).reshape(2, 3, 8, 8)
    b = pp.mmu_infer_batch(imgs, answers=["a cat", "a much longer answer about a dog"])
    T = b["input_ids"].shape[1]
    assert b["pixel_values"].shape == (2, 1, 3, 8, 8) and torch.equal(b["pixel_values"][:, 0], imgs)
    assert b["images_emb_mask"].shape == (2, 1, n_img) and bool(b["images_emb_mask"].all())
    assert int(b["images_seq_mask"].sum()) == int(b["images_emb_mask"].sum()) == 2 * n_img
    assert torch.equal(b["images_seq_mask"], b["input_ids"] == 5000)
    pad0 = int((b["attention_mask"][0] == 0).sum())
    assert pad0 > 0 and bool((b["input_ids"][0, :pad0] == 3).all()) and bool((b["attention_mask"][0, pad0:] == 1).all())
    assert int(b["attention_mask"][1].sum()) == T                      # the longest row has no padding


def test_write_png_round_trips_through_pil(tmp_path):
    import numpy as np
    from plangen_b200.prompts import write_png
    rng = np.random.default_rng(0)
    rgb = rng.integers(0, 256, (13, 7, 3), dtype=np.uint8)
    grey = rng.integers(0, 256, (5, 9), dtype=np.uint8)
    write_png(str(tmp_path / "a.png"), rgb)
    write_png(str(tmp_path / "g.png"), torch.from_numpy(grey))
    try:
        from PIL import Image
    except ImportError:
        pytest.skip("PIL not installed")
    assert np.array_equal(np.asarray(Image.open(tmp_path / "a.png")), rgb)
    assert np.array_equal(np.asarray(Image.open(tmp_path / "g.png")), grey)
    with pytest.raises(ValueError):
        write_png(str(tmp_path / "bad.png"), rgb.astype(np.float32))


# ------------------------------------------------------------------ torch custom-op layer (north_star: "thin C-ABI torch custom-op layer")
def test_custom_ops_are_registered_and_have_no_cpu_kernel():
    """Every hot-path C-ABI entry point is a torch.library operator in the `plangen_b200` namespace with a schema that
    names its mutated outputs; there is no CPU implementation to fall back to."""
    import plangen_b200.ops as ops
    from plangen_b200 import _lib
    for name in ops.OP_NAMES:
        op = getattr(torch.ops.plangen_b200, name)
        assert "!" in str(op.default._schema), name                      # declares what it writes
        assert "pg_" + name in _lib.EXPORTS, name                          # one C-ABI entry per operator
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.plangen_b200.images_to_u8(0, torch.zeros(4), torch.zeros(4, dtype=torch.uint8))
