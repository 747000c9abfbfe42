"""TEST / BENCH INFRASTRUCTURE -- never imported by the product.

Runs the UNMODIFIED reference (unpacked from oracle/_ref/reference.zip by oracle/refarchive.py) on the host CPUs
for bench.py's reference arm: the reference's own XSimGCL class, its own train() loop, its own sampler, losses,
encoder and torch.optim.Adam.  Harness-side shims only (SURVEY 8c; no edits to the reference):
  * cwd = a scratch directory (the reference writes ./log/),
  * Tensor.cuda / Module.cuda patched to identity (XSimGCL.py:24,46-47,73,90 hard-code .cuda()),
  * the batch generator the model imported is wrapped to time-stamp every batch and to stop after the requested
    number of steps, and fast_evaluation() is skipped (it is measured separately through test()).
"""
import importlib
import os
import random
import sys
import time

import numpy as np

TOP = ("base", "util", "data", "model")


def _conf(model, extra, d, B, lr, reg, topn):
    from util.conf import ModelConf
    c = ModelConf.__new__(ModelConf)
    c.config = {"training.set": "./synthetic/train.txt", "test.set": "./synthetic/test.txt", "model": {"name": model, "type": "graph"},
                "item.ranking.topN": list(topn), "embedding.size": d, "max.epoch": 1, "batch.size": B, "learning.rate": lr,
                "reg.lambda": reg, "output": "./results/", model: extra}
    return c


class ReferenceXSimGCL:
    """The reference's XSimGCL on a synthetic pair list (ids become the strings the reference expects)."""

    def __init__(self, ref_root, scratch, pair_users, pair_items, *, d, L, B, lr, reg, eps, tau, lam, l_star, test_users=1000):
        for k in [k for k in sys.modules if k.split(".")[0] in TOP]:
            del sys.modules[k]
        sys.path.insert(0, ref_root)
        os.makedirs(scratch, exist_ok=True)
        os.chdir(scratch)
        import torch
        self.torch = torch
        torch.Tensor.cuda = lambda self, *a, **k: self
        torch.nn.Module.cuda = lambda self, *a, **k: self
        self.mod = importlib.import_module("model.graph.XSimGCL")
        assert os.path.realpath(self.mod.__file__).startswith(os.path.realpath(ref_root))
        train = [[str(int(u)), str(int(i)), 1.0] for u, i in zip(pair_users, pair_items)]
        # a bounded test set: the first `test_users` users, one held-in item each (only its size matters for timing)
        seen, test = set(), []
        for u, i in zip(pair_users, pair_items):
            if u not in seen:
                seen.add(u)
                test.append([str(int(u)), str(int(i)), 1.0])
                if len(seen) >= test_users:
                    break
        conf = _conf("XSimGCL", {"n_layer": L, "l_star": l_star, "lambda": lam, "eps": eps, "tau": tau}, d, B, lr, reg, (10, 20))
        self.m = self.mod.XSimGCL(conf, train, test)
        self.m.fast_evaluation = lambda epoch: None
        self.m.best_user_emb = self.m.best_item_emb = None  # (set by fast_evaluation -> save() in a real run)
        self.B = B

    def time_steps(self, steps, warmup):
        """Seconds for `steps` iterations of the reference's train() loop after `warmup` (sampler included)."""
        torch = self.torch
        inner = importlib.import_module("util.sampler").next_batch_pairwise
        stamps = []

        def timed(data, batch_size, n_negs=1):
            for k, batch in enumerate(inner(data, batch_size, n_negs)):
                stamps.append(time.perf_counter())  # batch k handed over: step k-1 has finished
                if k >= warmup + steps:
                    return
                yield batch

        self.mod.next_batch_pairwise = timed
        self.m.maxEpoch = 1
        self.m.train()
        # stamps[k] .. stamps[k+1] = step k (forward, backward, Adam) + sampling of batch k+1
        return stamps[warmup + steps] - stamps[warmup]

    def time_rank(self):
        """(seconds, users, items) of one GraphRecommender.test() over the bounded test set."""
        torch = self.torch
        with torch.no_grad():
            self.m.user_emb, self.m.item_emb = self.m.model()
        self.m.test()  # first call: numba compiles find_k_largest (seconds); not part of the measurement
        t0 = time.perf_counter()
        rec = self.m.test()
        return time.perf_counter() - t0, len(rec), self.m.data.item_num
