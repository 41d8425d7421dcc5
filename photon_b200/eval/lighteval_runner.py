"""Offline runner for the reference's downstream-eval task lists (``conf/lighteval/*.txt``).

The reference ships those lists as input for the external ``lighteval`` CLI (a git dependency with accelerate / vllm extras,
ref: pyproject.toml:54,67; lines are ``suite|task|num_fewshot|truncate_fewshot``) and has no runner of its own. Neither the CLI nor
the HF hub is reachable here, so this module evaluates the same task lists against LOCAL jsonl copies of the datasets with the
scoring rules those tasks use, on any model of this framework (a server checkpoint ``.npz`` or a fresh model):

* multiple-choice tasks (hellaswag, arc, piqa, mmlu_pro, commonsense_qa, openbook_qa, winogrande) → length-normalised
  log-likelihood of every choice (``acc_norm``);
* generative tasks (trivia_qa, gsm8k, bbh) → greedy decoding + normalised exact match (gsm8k / bbh take the text after the
  last ``####`` / ``the answer is``);
* ``extended|ifeval`` needs instruction-following checkers that live in lighteval itself → reported as skipped.

Dataset rows use the ICL evaluator's schema (``photon_b200/eval/icl.py``): ``{"query", "choices", "gold"}`` for multiple choice,
``{"context", "answer", "aliases"}`` for generation; file = ``{data_root}/{task}.jsonl``. A missing file is reported as skipped, never
silently scored.

    python -m photon_b200.eval.lighteval_runner --tasks photon_b200/conf/lighteval/smollm2_base.txt --data-root ./eval_data \
        --model-config mpt-125m [--checkpoint runs/x/server/10/current_server_parameters.npz] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
from pathlib import Path
from typing import Any, Callable

import torch

from photon_b200.eval.icl import GenerateFn, ICLEvaluator

MULTIPLE_CHOICE = {"hellaswag", "arc", "piqa", "mmlu_pro", "commonsense_qa", "openbook_qa", "winogrande"}
GENERATIVE = {"trivia_qa": {}, "gsm8k": {"cot_delimiter": "####", "max_new_tokens": 256, "early_stopping_criteria": ["\n\n"]},
              "bbh": {"cot_delimiter": "the answer is", "max_new_tokens": 256, "early_stopping_criteria": ["\n\n"]}}


def parse_task_list(path: str | Path) -> list[dict[str, Any]]:
    """``suite|task|num_fewshot|truncate_fewshot`` lines (comments and blank lines ignored)."""
    out = []
    for raw in Path(path).read_text().splitlines():
        line = raw.split("#", 1)[0].strip()
        if not line:
            continue
        parts = line.split("|")
        if len(parts) != 4:
            raise ValueError(f"{path}: malformed task line {raw!r} (want suite|task|num_fewshot|truncate)")
        out.append({"suite": parts[0], "task": parts[1], "num_fewshot": int(parts[2]), "truncate_fewshot": bool(int(parts[3]))})
    return out


def to_icl_task(entry: dict[str, Any]) -> dict[str, Any] | None:
    """Task-list entry → an ICL task description, or None when the task type cannot be scored offline."""
    name = entry["task"]
    base = {"label": f"{entry['suite']}|{name}", "dataset_uri": f"{name}.jsonl", "num_fewshot": [entry["num_fewshot"]]}
    if name in MULTIPLE_CHOICE:
        return {**base, "icl_task_type": "multiple_choice", "continuation_delimiter": " "}
    if name in GENERATIVE:
        return {**base, "icl_task_type": "generation_task_with_answers", "continuation_delimiter": " ", **GENERATIVE[name]}
    return None


def run_task_list(tasks_file: str | Path, logits_fn: Callable[[torch.Tensor], torch.Tensor], tokenizer: Any, max_seq_len: int,
                  data_root: str | Path, generate_fn: GenerateFn | None = None) -> dict[str, Any]:
    """Score every entry of ``tasks_file``; ``generate_fn`` (a backend's ``generate``) batches the generative tasks."""
    ev = ICLEvaluator(logits_fn, tokenizer, max_seq_len, str(data_root), generate_fn=generate_fn)
    results: dict[str, Any] = {}
    for entry in parse_task_list(tasks_file):
        key = f"{entry['suite']}|{entry['task']}|{entry['num_fewshot']}"
        task = to_icl_task(entry)
        if task is None:
            results[key] = {"status": "skipped (needs lighteval's own checkers; not scorable offline)"}
            continue
        r = ev.evaluate_task(task)
        acc = next((v for k, v in r.items() if k.endswith("/accuracy")), None)
        results[key] = {"acc_norm" if entry["task"] in MULTIPLE_CHOICE else "exact_match": acc,
                        "n_samples": next((v for k, v in r.items() if k.endswith("/n_samples")), 0.0)} if acc is not None else r
    scored = [v[next(iter(v))] for v in results.values() if "status" not in v]
    results["all"] = {"average": sum(scored) / len(scored) if scored else None, "n_tasks_scored": len(scored), "n_tasks": len(results)}
    return results


def main() -> None:
    ap = argparse.ArgumentParser(prog="python -m photon_b200.eval.lighteval_runner")
    ap.add_argument("--tasks", required=True, help="task list, e.g. photon_b200/conf/lighteval/smollm2_base.txt")
    ap.add_argument("--data-root", required=True, help="directory with {task}.jsonl files")
    ap.add_argument("--model-config", default="mpt-125m", help="llm_config group name (mpt-125m / mpt-1b / mpt-3b / mpt-7b)")
    ap.add_argument("--checkpoint", default=None, help="npz / bin with the model's tensors in sorted-name order (server or centralised checkpoint)")
    ap.add_argument("--tokenizer", default="EleutherAI/gpt-neox-20b")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from photon_b200.config import compose
    from photon_b200.dataset.utils import build_tokenizer
    from photon_b200.models.mpt import MPTConfig, MPTForCausalLM
    from photon_b200.utils.core import load_model_parameters_from_file
    from photon_b200.utils.flat import FlatParams

    cfg = compose([f"llm_config={a.model_config}"])
    mcfg = MPTConfig.from_model_cfg(dict(cfg["llm_config"]["model"]))
    dev = torch.device("cuda" if torch.cuda.is_available() else "cpu")
    generate_fn = None
    if dev.type == "cuda":
        # the B200 engine: logits through its module view of the weights, generation KV-cached on its own kernels
        from photon_b200.train.backend import build_backend

        backend = build_backend(mcfg, dev, "amp_bf16", seed=17)
        if a.checkpoint:
            backend.flat.load_ndarrays(load_model_parameters_from_file(a.checkpoint)[: len(backend.flat.names)])
            backend.params_updated()
        backend.train_mode(False)
        logits_fn = backend.logits
        if getattr(backend, "can_generate", False):
            generate_fn = backend.generate
    else:
        if mcfg.attn_impl == "flash":
            mcfg.attn_impl = "torch"
        model = MPTForCausalLM(mcfg, device=dev, seed=17)
        if a.checkpoint:
            flat = FlatParams(model, device=dev, with_grad=False)
            flat.load_ndarrays(load_model_parameters_from_file(a.checkpoint)[: len(flat.names)])
        model.eval()

        @torch.no_grad()
        def logits_fn(ids: torch.Tensor) -> torch.Tensor:
            return model(ids.to(dev))

    res = run_task_list(a.tasks, logits_fn, build_tokenizer(a.tokenizer), mcfg.max_seq_len, a.data_root, generate_fn=generate_fn)
    text = json.dumps(res, indent=1)
    if a.out:
        Path(a.out).write_text(text)
    print(text)


if __name__ == "__main__":
    main()
