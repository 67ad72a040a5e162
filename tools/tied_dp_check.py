"""Multi-GPU parity check of the tied-embedding path (run under torchrun, NCCL): with a tied head (the lm_head matrix is also
the input embedding) the data-parallel step — row shards, the input-embedding term folded into each rank's gradient, one
exchange of the whole gradient, sharded AdamW, all-gather of the updated rows — must reproduce the single-GPU step on the
same global batch.  Two steps per mode: the second step's embedding lookup runs right after the first step's all-gather
was started, and its head asserts that the wait came first.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/tied_dp_check.py
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from rllm_b200 import transform as tf  # noqa: E402
from rllm_b200.backend import PolicyUpdateEngine, SyntheticTiedPolicyHead  # noqa: E402
from rllm_b200.config import AlgorithmConfig, PolicyLossConfig, TransformConfig  # noqa: E402
from rllm_b200.dp import DPContext  # noqa: E402
from rllm_b200.synth import WORKLOADS, make_episodes  # noqa: E402


class CheckedTiedHead(SyntheticTiedPolicyHead):
    engine: PolicyUpdateEngine | None = None

    def hidden_states(self, pb, db):
        assert not self.engine._weight_handles, "embedding lookup while the all-gather of the updated rows was pending"
        return super().hidden_states(pb, db)


def run(dp: DPContext, dev, episodes, groups, table, V, H, sharded, reuse=False, steps=2):
    """The body is a pure function of the token ids and W, and the pi_old / reference noise of the token id, so every
    sharding of the same batch sees the same per-token inputs."""
    cfg = PolicyLossConfig(loss_agg_mode="seq-mean-token-mean", clip_ratio_high=0.28, use_kl_loss=True, entropy_coeff=1e-3)
    policy = CheckedTiedHead(V, H, dev, seed=0, w_std=0.2)
    eng = PolicyUpdateEngine(policy, cfg, AlgorithmConfig(), dp=dp, chunk_tokens=2048, lr=1e-2)
    policy.engine = eng
    out = []
    for _ in range(steps):
        pb = eng.pack(episodes=episodes, sharded=sharded)
        db = eng.shard_to_device(pb)
        eng.old_log_probs(pb, db, groups=groups if reuse else None)
        db.old_logp = db.old_logp + 0.05 * table["n1"][db.labels.long()]
        db.ref_logp = db.old_logp + 0.1 * table["n2"][db.labels.long()]
        eng.advantages(pb, db, groups)
        eng.loss_weights(db)
        eng.forward_backward(pb, db)
        assert eng.last_compaction["forward"].startswith("reused") == bool(reuse), eng.last_compaction
        eng.reduce_gradients()
        sums = eng.reduce_metrics()
        grad = eng.reduced_gradient().clone()
        gnorm = eng.optimizer_step()  # sharded AdamW + all-gather of the bf16 rows under DP; left in flight for the next step
        out.append((dict(sums, grad_norm=gnorm), grad))
    eng.wait_weights()
    return out, policy.weight.clone()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--backend", default=None, choices=["nccl", "gloo"], help="default nccl; gloo lets the ranks share one GPU (parity of the algorithm, not of the NCCL exchange)")
    args = ap.parse_args()
    dp = DPContext.from_env(args.backend)
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    V, H = 4096, 256
    spec = WORKLOADS["qwen7b-solver-judge"]
    episodes = make_episodes(spec, seed=0, prompts=4, vocab=V)
    groups, _ = tf.transform_episodes_to_trajectory_groups(episodes, TransformConfig())
    g = torch.Generator(device=dev).manual_seed(11)
    table = {"n1": torch.randn(V, generator=g, device=dev), "n2": torch.randn(V, generator=g, device=dev)}
    modes = ("global pack", "shard-local pack", "shard-local pack + forward reuse", "global pack + forward reuse")
    results = {mode: run(dp, dev, episodes, groups, table, V, H, sharded=mode.startswith("shard-local pack"), reuse=mode.endswith("forward reuse")) for mode in modes}
    if dp.rank == 0:
        steps_1, w_1 = run(DPContext(), dev, episodes, groups, table, V, H, sharded=False)
        all_ok = True
        for mode, (steps_dp, w_dp) in results.items():
            for k, ((sums_dp, dw_dp), (sums_1, dw_1)) in enumerate(zip(steps_dp, steps_1)):
                rel = {n: abs(sums_dp[n] - sums_1[n]) / max(abs(sums_1[n]), 1e-12) for n in sums_1 if n != "grad_norm"}
                dw_err = float((dw_dp - dw_1).abs().max() / dw_1.abs().max())
                gn_err = abs(sums_dp["grad_norm"] - sums_1["grad_norm"]) / sums_1["grad_norm"]
                # step 2 runs on weights that may differ where step 1's gradient was ~0 (Adam moved them by ~lr * sign(g))
                tol_sum, tol_dw, tol_gn = (1e-6, 2e-2, 1e-4) if k == 0 else (1e-3, 5e-2, 1e-2)
                ok = all(v < tol_sum for v in rel.values()) and dw_err < tol_dw and gn_err < tol_gn
                all_ok &= ok
                print(json.dumps({"world_size": dp.world_size, "mode": mode, "step": k + 1, "ok": ok, "loss_dp": sums_dp["loss"], "loss_single": sums_1["loss"],
                                  "max_rel_sum_err": max(rel.values()), "dW_rel_err": dw_err, "grad_norm_rel_err": gn_err}), flush=True)
            w_same = float((w_dp == w_1).float().mean())  # Adam's first steps move by ~lr * sign(g): a gradient ~ 0 may flip
            all_ok &= w_same > 0.98
            print(json.dumps({"world_size": dp.world_size, "mode": mode, "weights_equal_after_two_steps": w_same}), flush=True)
        if not all_ok:
            sys.exit(1)
    dp.barrier()
    if dp.enabled:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
