"""Cost of training a tied-embedding model (the lm_head matrix is also the input embedding) on the qwen1.5b-gsm8k shape
(Qwen2.5-1.5B: H=1536, V=151936, tied): prints JSON lines.

  1. the fold kernel (rllm_b200_embedding_grad_accumulate) at the 1.5B shape on the workload's own input-stream length,
     uniform and Zipf ids: time (CUDA events, many launches), achieved GB/s from the algorithmic bytes, share of 7.7 TB/s;
  2. the host build of the fold order (input stream + counting sort) on the workload's shard;
  3. the policy-update step with a tied head against the same step with an untied head (same batch, same weights),
     alternated in one process.  The tied head's body backward is replaced by a fixed d_input_embeds tensor, so the
     difference is what the engine adds: the fold, the gradient exchange after the sweep instead of under it, the
     weight wait before the body.

    python tools/tied_bench.py                                   # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/tied_bench.py
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from rllm_b200 import loss as L  # noqa: E402
from rllm_b200 import transform as tf  # noqa: E402
from rllm_b200.backend import PolicyUpdateEngine, SyntheticPolicyHead, SyntheticTiedPolicyHead  # noqa: E402
from rllm_b200.config import AlgorithmConfig, PolicyLossConfig, TransformConfig  # noqa: E402
from rllm_b200.dp import DPContext  # noqa: E402
from rllm_b200.packing import token_segments  # noqa: E402
from rllm_b200.synth import WORKLOADS, make_episodes  # noqa: E402

HBM_BOUND_GBS = 7700.0  # HGX B200 data sheet, one GPU


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"gpu": q.stdout.strip()}


class FixedBackwardTiedHead(SyntheticTiedPolicyHead):
    """SyntheticTiedPolicyHead whose body backward hands back one precomputed d_input_embeds (the body's own cost is not
    the engine's)."""

    d_in: torch.Tensor | None = None

    def backward_hidden(self, d_hidden):
        if self.d_in is None:
            self.d_in = super().backward_hidden(d_hidden)
        return self.d_in


def fold_kernel(n_in: int, V: int, H: int, dev, iters: int) -> list[dict]:
    rng = np.random.default_rng(0)
    out = []
    for kind in ("uniform", "zipf"):
        ids = rng.integers(0, V, n_in).astype(np.int32) if kind == "uniform" else rng.permutation(((rng.zipf(1.2, n_in) - 1) % V)).astype(np.int32)
        seg = token_segments(ids, V)
        dseg = L.DeviceSegments.from_host(seg, dev)
        d_in = torch.randn(n_in, H, device=dev).to(torch.bfloat16)
        dw = torch.zeros(V, H, device=dev)
        for _ in range(3):
            L.embedding_grad_accumulate(d_in, dseg, dw)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            L.embedding_grad_accumulate(d_in, dseg, dw)
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / iters
        n_distinct = len(seg.seg_id)
        nbytes = n_in * H * 2 + n_distinct * H * 8 + seg.n_slots * H * 8
        out.append({"what": "fold_kernel", "ids": kind, "n_in": n_in, "H": H, "V": V, "n_distinct": n_distinct, "n_pieces": seg.n_pieces, "n_multi_segments": seg.n_multi,
                    "us": round(us, 2), "algorithmic_bytes": nbytes, "GBps": round(nbytes / us / 1e3, 1), "share_of_7.7TBps": round(nbytes / us / 1e3 / HBM_BOUND_GBS, 3),
                    "note": "inputs larger than L2 (d_in and the fp32 gradient rows); one launch = the two passes"})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the untied and tied arms")
    ap.add_argument("--kernel-iters", type=int, default=50)
    args = ap.parse_args()

    dp = DPContext.from_env()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    rank = dp.rank
    spec = WORKLOADS["qwen1.5b-gsm8k"]
    V, H = spec.vocab, spec.hidden
    episodes = make_episodes(spec, seed=0, prompts=spec.prompts, replicas=dp.world_size)  # bench.py's per-GPU batch for this workload
    groups, _ = tf.transform_episodes_to_trajectory_groups(episodes, TransformConfig())
    cfg = PolicyLossConfig(loss_agg_mode="seq-mean-token-mean", clip_ratio_low=0.2, clip_ratio_high=0.28)
    algo = AlgorithmConfig(estimator=spec.estimator)
    info = {"world_size": dp.world_size, **card()}

    arms = {}
    for name, head_cls in (("untied", SyntheticPolicyHead), ("tied", FixedBackwardTiedHead)):
        policy = head_cls(V, H, dev, seed=0)
        eng = PolicyUpdateEngine(policy, cfg, algo, dp=dp, max_response_length=spec.max_prompt_length + spec.max_response_length)
        eng.adaptive_balance = False  # the same partition for both arms
        pb = eng.pack(episodes=episodes, groups=groups, sharded=True)
        db = eng.shard_to_device(pb)
        hidden = policy.hidden_states(pb, db)
        eng.old_log_probs(pb, db, hidden)
        arms[name] = (eng, pb, db, hidden)

    eng_t, pb_t, db_t, _ = arms["tied"]
    if rank == 0:
        ids, _ = pb_t.input_stream(eng_t._shard_rows(pb_t, db_t))
        ts = []
        for _ in range(20):
            t0 = time.perf_counter()
            ids, _ = pb_t.input_stream(eng_t._shard_rows(pb_t, db_t))
            token_segments(ids, V)
            ts.append(time.perf_counter() - t0)
        print(json.dumps({"what": "host_segment_build", "n_in": len(ids), "rows": db_t.n_rows, "ms_median": round(1e3 * float(np.median(ts)), 3), "ms_min": round(1e3 * min(ts), 3),
                          "cpu": os.cpu_count(), **info}), flush=True)
        for r in fold_kernel(len(ids), V, H, dev, args.kernel_iters):
            print(json.dumps({**r, **info}), flush=True)
    dp.barrier()

    def step(eng, pb, db, hidden):
        eng.advantages(pb, db, groups)
        eng.loss_weights(db)
        eng.forward_backward(pb, db, hidden)
        eng.reduce_gradients()
        eng.reduce_metrics()
        eng.optimizer_step()

    def timed(name):
        eng, pb, db, hidden = arms[name]
        for _ in range(args.warmup):
            step(eng, pb, db, hidden)
        dp.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            step(eng, pb, db, hidden)
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / args.steps], dtype=torch.float64, device=dev)
        dp.all_reduce_max_(ms)
        return float(ms)

    res = {"untied": [], "tied": []}
    for _ in range(args.rounds):
        for name in ("untied", "tied"):
            res[name].append(timed(name))
    if rank == 0:
        u, t = float(np.median(res["untied"])), float(np.median(res["tied"]))
        print(json.dumps({"what": "step", "workload": spec.name, "tokens_per_rank": arms["tied"][2].n_tokens, "n_in_per_rank": arms["tied"][2].embed_segments.n_in,
                          "ms_untied": round(u, 3), "ms_tied": round(t, 3), "tied_over_untied": round(t / u, 4), "ms_untied_all": [round(x, 3) for x in res["untied"]],
                          "ms_tied_all": [round(x, 3) for x in res["tied"]], "note": "device step (advantages, loss weights, sweep, body backward fixed, fold, exchange, metrics, optimizer); max over ranks; median of the alternations",
                          **info}), flush=True)
    dp.barrier()
    if dp.enabled:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
