"""In-context-learning evaluation + Eval Gauntlet aggregation.

The reference gets these from llm-foundry (``build_evaluators`` / ``EvalGauntlet``; wired at
photon/centralised_train.py:120-136 and photon/clients/trainer_utils.py) and ships only the task
tables (``conf/icl_tasks_config/*.yaml``, ``conf/eval_gauntlet_config/*.yaml``).  This module is a
self-contained implementation of the two task types that dominate those tables:

* ``language_modeling``   — exact-match of the greedy continuation (teacher-forced argmax);
* ``multiple_choice``     — pick the choice with the highest length-normalised log-likelihood;
  ``schema`` tasks are scored the same way with the context varying instead of the continuation.

* ``generation_task_with_answers`` — greedy decoding until ``max_new_tokens`` or an ``early_stopping_criteria`` string;
  exact match against any of the ``answer`` / ``aliases`` after llm-foundry's normalisation (lower-case, punctuation and
  articles stripped) unless ``do_normalization: false``; with a ``cot_delimiter`` only the text after it counts. With a
  ``generate_fn`` (a backend's ``generate``: on the B200 engine, KV-cached decoding on its own kernels) the rows are
  generated ``batch_size`` at a time; without one, row by row with one ``logits_fn`` call per new token.

Datasets are jsonl files resolved against ``icl_tasks_config.root_dir`` (there is no network, so missing files yield
``skipped``).
"""
from __future__ import annotations

import json
from pathlib import Path
from typing import Any, Callable

import torch

TASK_DEFAULTS = {"num_fewshot": [0], "continuation_delimiter": " ", "example_delimiter": "\n", "prompt_string": "",
                 "question_prelimiter": "", "batch_size": 4, "max_new_tokens": 64, "early_stopping_criteria": [],
                 "cot_delimiter": "", "do_normalization": True}


def expand_task(task: dict[str, Any]) -> dict[str, Any]:
    """Fill the defaults omitted by the compact task tables."""
    t = {**TASK_DEFAULTS, **task}
    if isinstance(t["num_fewshot"], int):
        t["num_fewshot"] = [t["num_fewshot"]]
    if "label" not in t or "dataset_uri" not in t or "icl_task_type" not in t:
        raise ValueError(f"ICL task needs label/dataset_uri/icl_task_type: {task}")
    return t


def _normalize_answer(text: str) -> str:
    """llm-foundry's exact-match normalisation: lower-case, drop punctuation and articles, squeeze whitespace."""
    import re
    import string

    text = "".join(ch for ch in text.lower() if ch not in set(string.punctuation))
    return " ".join(re.sub(r"\b(a|an|the)\b", " ", text).split())


def _rows(path: Path) -> list[dict[str, Any]]:
    return [json.loads(l) for l in path.read_text().splitlines() if l.strip()]


GenerateFn = Callable[[list[list[int]], int, "int | None", "Callable[[int, list[int]], bool] | None"], list[list[int]]]


def _cut_at_stop(text: str, stops: list[str]) -> str | None:
    """``text`` up to the earliest stop string, or None when no stop string occurs."""
    hit = [text.index(s) for s in stops if s and s in text]
    return text[: min(hit)] if hit else None


class ICLEvaluator:
    """``logits_fn(ids [B,S] LongTensor) -> [B,S,V]`` abstracts the model (torch backend or engine).

    ``generate_fn(prompts, max_new_tokens, eos_id, stop) -> new ids per prompt`` (optional): batched greedy decoding for the
    generation tasks, ``stop(row, new_ids) -> bool`` ending a row; the backends' ``generate`` has this signature."""

    def __init__(self, logits_fn: Callable[[torch.Tensor], torch.Tensor], tokenizer: Any, max_seq_len: int, root_dir: str | None = None,
                 generate_fn: GenerateFn | None = None) -> None:
        self.logits_fn, self.tok, self.max_seq_len, self.root = logits_fn, tokenizer, int(max_seq_len), Path(root_dir or ".")
        self.generate_fn = generate_fn

    def _enc(self, text: str) -> list[int]:
        if hasattr(self.tok, "encode") and not hasattr(self.tok, "__call__"):
            return self.tok.encode(text)
        return self.tok(text, add_special_tokens=False)["input_ids"] if callable(self.tok) else self.tok.encode(text)

    def _fewshot_prefix(self, rows: list[dict[str, Any]], idx: int, k: int, t: dict[str, Any]) -> str:
        shots = [r for i, r in enumerate(rows) if i != idx][:k]
        parts = []
        for r in shots:
            cont = r.get("continuation", r["choices"][r["gold"]] if "choices" in r else "")
            parts.append(f"{t['question_prelimiter']}{r.get('context', r.get('query', ''))}{t['continuation_delimiter']}{cont}")
        return t["prompt_string"] + t["example_delimiter"].join(parts) + (t["example_delimiter"] if parts else "")

    @torch.no_grad()
    def _continuation_stats(self, ctx: list[int], cont: list[int]) -> tuple[float, bool]:
        """(sum log p(cont | ctx), greedy-exact-match) with left truncation to ``max_seq_len``."""
        ids = (ctx + cont)[-self.max_seq_len:]
        n = min(len(cont), len(ids) - 1)
        x = torch.tensor([ids], dtype=torch.long)
        logp = torch.log_softmax(self.logits_fn(x)[0].float(), dim=-1)
        pos = torch.arange(len(ids) - n - 1, len(ids) - 1)
        tgt = torch.tensor(ids[-n:])
        lp = logp[pos].cpu()
        return float(lp[torch.arange(n), tgt].sum()), bool((lp.argmax(-1) == tgt).all())

    @torch.no_grad()
    def _generate(self, ctx: list[int], max_new_tokens: int, stops: list[str]) -> str:
        """Greedy continuation of ``ctx`` as text, cut at the first stop string."""
        ids, new = list(ctx), []
        eos = getattr(self.tok, "eos_token_id", None)
        for _ in range(max_new_tokens):
            window = ids[-self.max_seq_len:]
            nxt = int(self.logits_fn(torch.tensor([window], dtype=torch.long))[0, -1].float().argmax())
            if eos is not None and nxt == eos:
                break
            ids.append(nxt), new.append(nxt)
            cut = _cut_at_stop(self.tok.decode(new), stops)
            if cut is not None:
                return cut
        return self.tok.decode(new)

    def _generate_batch(self, ctxs: list[list[int]], max_new_tokens: int, stops: list[str]) -> list[str]:
        """:meth:`_generate` for many prompts in one ``generate_fn`` call: the same texts, stop strings checked on the decoded
        text of each row after every token."""
        stop = (lambda r, new: _cut_at_stop(self.tok.decode(new), stops) is not None) if any(stops) else None
        outs = self.generate_fn(ctxs, max_new_tokens, getattr(self.tok, "eos_token_id", None), stop)
        texts = [self.tok.decode(o) for o in outs]
        return [t if (c := _cut_at_stop(t, stops)) is None else c for t in texts]

    @staticmethod
    def _score_generation(text: str, row: dict[str, Any], t: dict[str, Any]) -> int:
        """1 when the generated ``text`` (after ``cot_delimiter``) matches the answer or an alias, else 0."""
        if t["cot_delimiter"] and t["cot_delimiter"] in text:
            text = text.split(t["cot_delimiter"])[-1]
        golds = [str(row["answer"])] + [str(a) for a in row.get("aliases", [])]
        norm = _normalize_answer if t["do_normalization"] else (lambda x: x.strip())
        return int(any(norm(text).startswith(norm(g)) for g in golds if norm(g)))

    def _generation_prompt(self, rows: list[dict[str, Any]], i: int, k: int, t: dict[str, Any]) -> list[int]:
        return self._enc(self._fewshot_prefix(rows, i, k, t) + t["question_prelimiter"] + rows[i]["context"] + t["continuation_delimiter"].rstrip())

    def evaluate_task(self, task: dict[str, Any]) -> dict[str, float | str]:
        t = expand_task(task)
        path = self.root / t["dataset_uri"]
        if not path.exists():
            return {"status": "skipped (dataset missing offline)"}
        kind = t["icl_task_type"]
        if kind not in ("language_modeling", "multiple_choice", "schema", "generation_task_with_answers"):
            return {"status": f"unsupported task type {kind}"}
        if kind == "generation_task_with_answers" and not hasattr(self.tok, "decode"):
            return {"status": "generation tasks need a tokenizer with decode()"}
        rows = _rows(path)
        out: dict[str, float | str] = {}
        stops = list(t["early_stopping_criteria"] or [])
        batched = kind == "generation_task_with_answers" and self.generate_fn is not None
        for k in t["num_fewshot"]:
            correct = 0
            bs = max(1, int(t["batch_size"]))
            for lo in range(0, len(rows), bs) if batched else ():
                ctxs = [self._generation_prompt(rows, i, k, t) for i in range(lo, min(lo + bs, len(rows)))]
                texts = self._generate_batch(ctxs, int(t["max_new_tokens"]), stops)
                correct += sum(self._score_generation(text, rows[lo + j], t) for j, text in enumerate(texts))
            for i, r in enumerate(rows if not batched else ()):
                prefix = self._fewshot_prefix(rows, i, k, t)
                if kind == "generation_task_with_answers":
                    text = self._generate(self._generation_prompt(rows, i, k, t), int(t["max_new_tokens"]), stops)
                    correct += self._score_generation(text, r, t)
                elif kind == "language_modeling":
                    ctx = self._enc(prefix + t["question_prelimiter"] + r["context"] + t["continuation_delimiter"].rstrip())
                    _, em = self._continuation_stats(ctx, self._enc(" " + r["continuation"].lstrip()))
                    correct += int(em)
                else:
                    scores = []
                    if kind == "multiple_choice":
                        ctx = self._enc(prefix + t["question_prelimiter"] + r["query"] + t["continuation_delimiter"].rstrip())
                        for ch in r["choices"]:
                            cont = self._enc(" " + ch.lstrip())
                            scores.append(self._continuation_stats(ctx, cont)[0] / max(1, len(cont)))
                    else:  # schema: the context options vary, the continuation is shared
                        cont = self._enc(" " + r["continuation"].lstrip())
                        for opt in r["context_options"]:
                            scores.append(self._continuation_stats(self._enc(prefix + opt), cont)[0] / max(1, len(cont)))
                    correct += int(int(torch.tensor(scores).argmax()) == int(r["gold"]))
            out[f"{t['label']}/{k}-shot/accuracy"] = correct / max(1, len(rows))
            out[f"{t['label']}/{k}-shot/n_samples"] = float(len(rows))
        return out


class EvalGauntlet:
    """Category averages over benchmark accuracies with random-baseline subtraction and rescaling
    (the semantics of llm-foundry's EvalGauntlet for ``weighting: EQUAL``)."""

    def __init__(self, cfg: dict[str, Any]) -> None:
        self.cfg = cfg
        if cfg.get("weighting", "EQUAL") not in ("EQUAL", "SAMPLE_SZ", "LOG_SAMPLE_SZ"):
            raise ValueError(f"unknown eval_gauntlet weighting {cfg.get('weighting')!r} (EQUAL | SAMPLE_SZ | LOG_SAMPLE_SZ)")

    def _weight(self, n_samples: float) -> float:
        """llm-foundry's benchmark weights inside a category: equal, by sample count, or by log2 of it (at least 1)."""
        import math

        mode = self.cfg.get("weighting", "EQUAL")
        if mode == "EQUAL" or n_samples <= 0:
            return 1.0
        return float(n_samples) if mode == "SAMPLE_SZ" else max(math.log2(n_samples), 1.0)

    def aggregate(self, metrics: dict[str, float]) -> dict[str, float]:
        out: dict[str, float] = {}
        for cat in self.cfg.get("categories", []):
            vals, wts = [], []
            for b in cat["benchmarks"]:
                key = f"{b['name']}/{b['num_fewshot']}-shot/accuracy"
                if key not in metrics:
                    continue
                wts.append(self._weight(float(metrics.get(f"{b['name']}/{b['num_fewshot']}-shot/n_samples", 0.0))))
                acc, base = float(metrics[key]), float(b.get("random_baseline", 0.0))
                if self.cfg.get("subtract_random_baseline", True):
                    acc -= base
                if self.cfg.get("rescale_accuracy", True) and base < 1.0:
                    acc /= (1.0 - base)
                vals.append(acc)
            if vals:
                out[f"icl/metrics/eval_gauntlet/{cat['name']}"] = sum(v * w for v, w in zip(vals, wts)) / sum(wts)
        for name, cats in (self.cfg.get("averages") or {}).items():
            vs = [out[f"icl/metrics/eval_gauntlet/{c}"] for c in cats if f"icl/metrics/eval_gauntlet/{c}" in out]
            if vs:
                out[f"icl/metrics/eval_gauntlet/{name}"] = sum(vs) / len(vs)
        return out


def run_icl_suite(logits_fn: Callable[[torch.Tensor], torch.Tensor], tokenizer: Any, cfg: Any, max_seq_len: int,
                  generate_fn: GenerateFn | None = None) -> dict[str, Any]:
    """Evaluate every task of ``cfg.icl_tasks_config`` and fold through ``cfg.eval_gauntlet_config``; ``generate_fn``
    batches the generation tasks (see :class:`ICLEvaluator`)."""
    icl = cfg.get("icl_tasks_config") or {}
    tasks = icl.get("icl_tasks") or []
    ev = ICLEvaluator(logits_fn, tokenizer, max_seq_len, icl.get("root_dir"), generate_fn=generate_fn)
    metrics: dict[str, Any] = {}
    for t in tasks:
        metrics.update({k: v for k, v in ev.evaluate_task(dict(t)).items() if not (k == "status")})
    g = (cfg.get("eval_gauntlet_config") or {}).get("eval_gauntlet")
    if g:
        metrics.update(EvalGauntlet(dict(g)).aggregate({k: v for k, v in metrics.items() if isinstance(v, float)}))
    return metrics
