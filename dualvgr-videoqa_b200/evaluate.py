"""Validation path on the device — the loop body of the reference's validate.py:44-134 restated B200-first.

  * eval-mode forward through the same fused path as training; under torch.no_grad() the unit stack keeps no fp32 copies of
    the graph outputs and computes no auxiliary terms (the 7-tuple's per-layer lists are bf16 views nobody reads)
  * preds = argmax, agreeings, and the per-question-type (MSVD / MSRVTT: first question word, validate.py:66-80) or
    per-category (SVQA: question_categories, validate.py:97-130) counters in ONE kernel per batch (dvgr_accuracy_counters):
    no Python loop over the batch, no host sync per sample; the host reads [n_cat + 1, 2] int64 once at the end
  * optionally the whole eval step (forward + counters) replayed as a CUDA graph on static input buffers."""
import torch

from . import ops

MSVD_TYPES = ("what", "who", "how", "when", "where")                      # validate.py:66-80
SVQA_CATEGORIES = ("count", "exist", "query_color", "query_size", "query_actiontype", "query_direction", "query_shape",
                   "compare_more", "compare_equal", "compare_less", "attribute_compare_color", "attribute_compare_size",
                   "attribute_compare_actiontype", "attribute_compare_direction", "attribute_compare_shape")


class EvalEngine:
    def __init__(self, model, categories, question_token_to_idx=None):
        """categories: names of the accuracy groups. With question_token_to_idx the group of a sample is decided by its first
        question token (groups = words such as 'what', 'who', ...); otherwise by the category id passed to step()."""
        self.model = model
        self.categories = tuple(categories)
        dev = next(model.parameters()).device
        self.counts = torch.zeros((len(self.categories) + 1, 2), dtype=torch.int64, device=dev)
        self.token_to_cat = None
        if question_token_to_idx is not None:
            V = max(question_token_to_idx.values()) + 1
            table = torch.full((V,), -1, dtype=torch.int32)
            for c, word in enumerate(self.categories):
                if word in question_token_to_idx:
                    table[question_token_to_idx[word]] = c
            self.token_to_cat = table.to(dev)
        self.graph = None

    def reset(self):
        self.counts.zero_()

    @torch.no_grad()
    def step(self, app, mot, question, question_len, answers, question_categories=None, want_preds=False):
        """One validation batch: returns (logits, preds | None); the counters accumulate on the device."""
        self.model.eval()
        return self._count(self.model(app, mot, question, question_len)[0], question, answers, question_categories,
                           want_preds)

    @torch.no_grad()
    def step_from_store(self, dstore, rows, question, question_len, answers, question_categories=None, want_preds=False):
        """step() on the batch (dstore.app[rows], dstore.mot[rows]) of a device-resident feature store
        (loader.DeviceFeatureStore), gathered inside the input prologue kernels; rows [B] int32 on the device. A row
        outside [0, V) sets dstore.err (read it with dstore.read_error())."""
        self.model.eval()
        return self._count(self.model.forward_from_store(dstore, rows, question, question_len)[0], question, answers,
                           question_categories, want_preds)

    def _count(self, logits, question, answers, question_categories, want_preds):
        preds = ops.accuracy_counters(logits, answers.reshape(-1), self.counts,
                                      category=question_categories.reshape(-1) if question_categories is not None else None,
                                      tokens=question if (question_categories is None and self.token_to_cat is not None) else None,
                                      token_to_cat=self.token_to_cat, want_preds=want_preds)
        return logits, preds

    def capture(self, app, mot, question, question_len, answers, question_categories=None):
        """Records the eval step as a CUDA graph over static input buffers (load_batch + replay afterwards)."""
        def step(st):
            return self.step(st["app"], st["mot"], st["q"], st["qlen"], st["ans"], st.get("cat"))
        return self._capture(dict(app=app, mot=mot, q=question, qlen=question_len, ans=answers), question_categories, step)

    def capture_from_store(self, dstore, rows, question, question_len, answers, question_categories=None):
        """capture() for step_from_store: static inputs are the rows and the question / answer (/ category) tensors only;
        load_rows + replay afterwards. The graph has the batch size of `rows`: run a shorter last batch through
        step_from_store."""
        def step(st):
            return self.step_from_store(dstore, st["rows"], st["q"], st["qlen"], st["ans"], st.get("cat"))
        return self._capture(dict(rows=rows, q=question, qlen=question_len, ans=answers), question_categories, step)

    def _capture(self, named, question_categories, step):
        if question_categories is not None:
            named["cat"] = question_categories
        self.static = {k: v.clone() for k, v in named.items()}
        st = self.static
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        saved = self.counts.clone()
        with torch.cuda.stream(side):
            for _ in range(2):
                step(st)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_logits, _ = step(st)
        self.counts.copy_(saved)                      # warm-up and capture must not count
        return self.graph

    def load_batch(self, **tensors):
        for k, v in tensors.items():
            self.static[k].copy_(v, non_blocking=True)

    def load_rows(self, rows, question, question_len, answers, question_categories=None):
        """The next full batch of a capture_from_store() graph."""
        named = dict(rows=rows, q=question, qlen=question_len, ans=answers)
        if question_categories is not None:
            named["cat"] = question_categories
        self.load_batch(**named)

    def replay(self):
        self.graph.replay()
        return self.static_logits

    def result(self):
        """{'all': acc, category: acc, ...} plus raw counts — the ONE host read of the validation loop."""
        c = self.counts.cpu()
        out = {"counts": {name: (int(c[i, 0]), int(c[i, 1])) for i, name in enumerate(self.categories)}}
        out["counts"]["all"] = (int(c[-1, 0]), int(c[-1, 1]))
        for name, (ok, n) in out["counts"].items():
            out[name] = ok / n if n else 0.0
        return out
