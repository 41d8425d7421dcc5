"""Batched greedy generation on the stock backend and the evaluators that use it: ``TorchBackend.generate`` must give exactly
the tokens of the per-row recompute path (``ICLEvaluator._generate``), and batching the generation tasks through a
``generate_fn`` must not change any score."""
import json
import math
from types import SimpleNamespace

import pytest
import torch

from photon_b200.dataset.utils import ByteTokenizer
from photon_b200.eval import ICLEvaluator
from photon_b200.models.mpt import MPTConfig
from photon_b200.train.backend import TorchBackend

MSL = 64


class CharTok:
    """One distinct character per id, so a stop string can name any single token."""

    def __init__(self, eos_token_id=None):
        self.eos_token_id = eos_token_id

    def encode(self, text):
        return [ord(ch) - 0x4E00 for ch in text]

    def decode(self, ids):
        return "".join(chr(0x4E00 + int(i)) for i in ids)


@pytest.fixture(scope="module")
def tiny():
    cfg = MPTConfig(d_model=64, n_heads=2, n_layers=2, max_seq_len=MSL, vocab_size=128, attn_impl="torch")
    be = TorchBackend(cfg, device="cpu", precision="fp32", seed=3)
    be.train_mode(False)
    return be


def _prompts():
    g = torch.Generator().manual_seed(11)
    lens = [1, 5, 17, 33, 60]          # ragged; 60 + new tokens crosses max_seq_len = 64
    return [torch.randint(1, 128, (n,), generator=g).tolist() for n in lens]


def _per_row(be, tok, prompts, n_new, stops):
    ev = ICLEvaluator(be.logits, tok, MSL)
    return [ev._generate(p, n_new, stops) for p in prompts]   # noqa: SLF001


def test_batched_generate_matches_per_row_recompute(tiny):
    tok = CharTok()
    prompts = _prompts()
    want = _per_row(tiny, tok, prompts, 12, [])
    got = tiny.generate(prompts, 12)
    assert [tok.decode(g) for g in got] == want
    assert all(len(g) == 12 for g in got)


def test_batched_generate_eos_and_stop_string(tiny):
    prompts = _prompts()
    free = tiny.generate(prompts, 12)
    eos = free[1][4]                                   # row 1 ends before its 5th token (or earlier, if it occurs sooner)
    stop_tok = free[3][2]                              # row 3 stops once this token has been generated
    tok = CharTok(eos_token_id=eos)
    stops = [tok.decode([stop_tok])]
    want = _per_row(tiny, tok, prompts, 12, stops)
    ev = ICLEvaluator(tiny.logits, tok, MSL, generate_fn=tiny.generate)
    assert ev._generate_batch(prompts, 12, stops) == want   # noqa: SLF001
    raw = tiny.generate(prompts, 12, eos_id=eos, stop=lambda r, new: any(s in tok.decode(new) for s in stops))
    assert eos not in sum(raw, []) and len(raw[1]) <= 4
    assert len(raw[3]) <= 3 and tok.decode(raw[3]).endswith(stops[0])


def test_generate_window_beyond_max_seq_len(tiny):
    """A 60-token prompt with 12 new tokens runs past max_seq_len = 64: the batched path continues over the last 64 ids, and a
    prompt longer than max_seq_len is left-truncated, exactly as the recompute path does."""
    tok = CharTok()
    g = torch.Generator().manual_seed(5)
    prompts = [torch.randint(1, 128, (60,), generator=g).tolist(), torch.randint(1, 128, (90,), generator=g).tolist(), [7]]
    assert [tok.decode(x) for x in tiny.generate(prompts, 12)] == _per_row(tiny, tok, prompts, 12, [])
    assert tiny.generate(prompts, 0) == [[], [], []]


def _fake_logits(ids):
    """The byte-successor 'model' of test_eval_icl: next byte = current byte + 1."""
    B, S = ids.shape
    out = torch.full((B, S, 257), -10.0)
    out[torch.arange(B)[:, None], torch.arange(S)[None], (ids + 1) % 257] = 10.0
    return out


def _fake_generate(logits_fn, max_seq_len):
    """The stock backend's batched recompute over a fake model."""
    fake = SimpleNamespace(cfg=SimpleNamespace(max_seq_len=max_seq_len), logits=logits_fn)
    return lambda *a, **k: TorchBackend.generate(fake, *a, **k)


@pytest.mark.parametrize("batch_size", [1, 3, 64])
def test_icl_generation_scores_unchanged_by_batching(tmp_path, batch_size):
    rows = [{"context": "a", "answer": "BCD"}, {"context": "a", "answer": "zz", "aliases": ["bcd"]}, {"context": "k", "answer": "nope"},
            {"context": "wxy", "answer": "z{"}, {"context": "mn", "answer": "opq"}, {"context": "abcdefgh", "answer": "ij"},
            {"context": "r", "answer": "st", "aliases": ["xx"]}]
    (tmp_path / "gen.jsonl").write_text("\n".join(json.dumps(r) for r in rows))
    (tmp_path / "cot.jsonl").write_text("\n".join(json.dumps(r) for r in [{"context": "a", "answer": "fg"}, {"context": "p", "answer": "uv"},
                                                                          {"context": "b", "answer": "zz"}]))
    tok = ByteTokenizer()
    tasks = [{"label": "gen", "dataset_uri": "gen.jsonl", "icl_task_type": "generation_task_with_answers", "num_fewshot": [0, 1],
              "continuation_delimiter": "", "early_stopping_criteria": ["e"], "max_new_tokens": 8, "batch_size": batch_size},
             {"label": "cot", "dataset_uri": "cot.jsonl", "icl_task_type": "generation_task_with_answers", "continuation_delimiter": "",
              "cot_delimiter": "e", "early_stopping_criteria": ["h", "x"], "max_new_tokens": 10, "do_normalization": False,
              "batch_size": batch_size}]
    plain = ICLEvaluator(_fake_logits, tok, 64, str(tmp_path))
    batched = ICLEvaluator(_fake_logits, tok, 64, str(tmp_path), generate_fn=_fake_generate(_fake_logits, 64))
    for t in tasks:
        want, got = plain.evaluate_task(dict(t)), batched.evaluate_task(dict(t))
        assert got == want
        assert any(0.0 < v < 1.0 for k, v in want.items() if k.endswith("/accuracy")), want   # the fixture separates rows
        assert all(v == float(len(rows) if t["label"] == "gen" else 3) for k, v in want.items() if k.endswith("/n_samples"))


def test_lighteval_generative_tasks_with_generate_fn(tmp_path):
    from photon_b200.eval.lighteval_runner import run_task_list

    class Tok:
        eos_token_id = None

        def encode(self, text):
            return list(text.encode())

        def decode(self, ids):
            return bytes(ids).decode(errors="ignore")

    def logits_fn(ids):
        B, S = ids.shape
        out = torch.full((B, S, 256), -10.0)
        out[torch.arange(B)[:, None], torch.arange(S)[None, :], (ids + 1) % 256] = 10.0
        return out

    (tmp_path / "trivia_qa.jsonl").write_text("\n".join(json.dumps(r) for r in [
        {"context": "ab", "answer": "cde", "aliases": []}, {"context": "x", "answer": "q", "aliases": ["yz"]}, {"context": "k", "answer": "no"}]))
    (tmp_path / "gsm8k.jsonl").write_text("\n".join(json.dumps(r) for r in [{"context": "a", "answer": "bcd"}, {"context": "0", "answer": "9"}]))
    tasks = tmp_path / "tasks.txt"
    tasks.write_text("custom|trivia_qa|0|1\ncustom|gsm8k|1|1\n")
    want = run_task_list(tasks, logits_fn, Tok(), 64, tmp_path)
    got = run_task_list(tasks, logits_fn, Tok(), 64, tmp_path, generate_fn=_fake_generate(logits_fn, 64))
    assert got == want
    assert math.isclose(want["custom|trivia_qa|0"]["exact_match"], 2 / 3)
