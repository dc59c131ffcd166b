"""Stage-2 caller (SURVEY section 8f, rank 3): rank the retrieved candidates with the LLM without ever forming
the [B, T, V] logits.

The reference's patched forward projects ALL T positions onto ALL V tokens, widens to fp32 and then keeps
`[:, -1]` (model/llm.py:102-131); the trainer / demo feed that row to `ManualVerbalizer.process_logits`
(trainer/llm.py:63-72 via HF's numpy round trip, demo/inference.py:56-76 via `.to("cpu")`).  Here the
transformer body runs as it is (library code, out of scope), and its last-position hidden state goes
straight into the fused label-row kernel (`ManualVerbalizer.score_hidden` -> lrb_verbalizer_score); the
metrics stay on the device.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import torch

from .metrics import absolute_recall_mrr_ndcg_for_ks
from .verbalizer import ManualVerbalizer


def _body(llm):
    body = getattr(llm, "model", None)
    if body is None or not hasattr(llm, "lm_head"):
        raise TypeError("expected a causal LM with `.model` (transformer body) and `.lm_head` "
                        "(LlamaForCausalLM / LlamaForCausalLMPatched, model/llm.py:17)")
    return body


@torch.no_grad()
def score_candidates(llm, verbalizer: ManualVerbalizer, input_ids: torch.Tensor,
                     attention_mask: Optional[torch.Tensor] = None, **body_kwargs) -> torch.Tensor:
    """[B, T] prompt ids -> [B, C] label scores (C = number of candidate letters).

    Equals `verbalizer.process_logits(llm(input_ids, attention_mask).logits[:, -1])` of the reference in eval
    mode (model/llm.py:113-114,131; trainer/verb.py:546-586) up to the bf16 rounding of the 20 logits."""
    hidden = _body(llm)(input_ids=input_ids, attention_mask=attention_mask, **body_kwargs)[0]   # [B, T, H]
    return verbalizer.score_hidden(hidden[:, -1], llm.lm_head.weight,
                                   round_logits_to_bf16=llm.lm_head.weight.dtype == torch.bfloat16)


@torch.no_grad()
def rank_candidates(llm, tokenizer, prompt: str, candidates: Sequence[int], verbalizer: ManualVerbalizer,
                    top_k: int = 10) -> List[int]:
    """demo/inference.py:56-76 with the scores computed on the device."""
    dev = llm.lm_head.weight.device
    inputs = tokenizer(prompt, return_tensors="pt").to(dev)
    scores = score_candidates(llm, verbalizer, inputs["input_ids"], inputs.get("attention_mask"))
    order = torch.topk(scores, min(top_k, scores.shape[1])).indices[0].tolist()
    return [candidates[i] for i in order]


@torch.no_grad()
def rerank_metrics(scores: torch.Tensor, labels: torch.Tensor, ks: Sequence[int]) -> Dict[str, float]:
    """`compute_metrics_for_ks(ks, verbalizer)` (trainer/llm.py:63-72) for label scores that are already on the
    device: Recall/MRR/NDCG@ks of the label index among the C candidates, same keys as the reference.

    Ties are ranked by (score desc, index asc), the merge kernel's order: the label's 0-based rank is the number of
    candidates with a higher score plus the tied ones with a lower index.  bf16-rounded label logits tie exactly
    quite often; the reference's `(-scores).argsort()` leaves the order of ties undefined."""
    return absolute_recall_mrr_ndcg_for_ks(scores, labels.view(-1), list(ks))


# ---- the demo's retriever artefact (setup_demo.py:46-47, demo/inference.py:20-23,46-53) ------------------------------
def export_retriever(model, path: str) -> None:
    """What `torch.jit.script(model).save("demo/retriever.pth")` is to the reference demo (setup_demo.py:46-47): one
    file the demo can load without the training code.  The kernels are reached through a C ABI, which TorchScript
    cannot trace, so the artefact is the model's hyper-parameters + `state_dict` (the reference's own keys and dtypes);
    `load_retriever` rebuilds the `LRURec` from it."""
    args = model.args
    keep = {k: getattr(args, k) for k in ("num_items", "bert_hidden_units", "bert_num_blocks", "bert_dropout",
                                           "bert_attn_dropout") if hasattr(args, k)}
    torch.save({"format": "llamarec_b200.retriever.v1", "args": keep,
                "state_dict": {k: v.detach().cpu() for k, v in model.state_dict().items()}}, path)


def load_retriever(path: str = "retriever.pth", device: str = "cuda"):
    """demo/inference.py:20-23 -- load the exported retriever, in eval mode, on `device`."""
    from types import SimpleNamespace
    from .model import LRURec
    blob = torch.load(path, map_location="cpu", weights_only=False)
    if blob.get("format") != "llamarec_b200.retriever.v1":
        raise ValueError(f"{path} is not a llamarec_b200 retriever export")
    model = LRURec(SimpleNamespace(**blob["args"]))
    model.load_state_dict(blob["state_dict"])
    return model.to(device).eval()


def retrieve_candidates(model, query: Sequence[int], top_k: int = 20) -> List[int]:
    """demo/inference.py:46-53: `topk(model(seqs)[:, -1, :], top_k)` for one interaction history, without the history
    mask (the demo does not apply one) and without the [1, L, N+1] score tensor."""
    query = list(query)
    if not query:
        raise ValueError("retrieve_candidates needs at least one interaction")
    seqs = torch.tensor(query, dtype=torch.int64).unsqueeze(0)
    return model.retrieve(seqs, k=top_k, exclude_history=False)["ids"][0].tolist()
