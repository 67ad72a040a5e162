"""bench.py — policy-update tokens/sec of the B200-native GRPO path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (N>1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the reference's path as ported by oracle/
    python bench.py ... --dump-outputs DIR                    # + DIR/<name>.npy: what the last timed update step computed

Workload (config.workload): the headline config ``configs[2]`` — Qwen2.5-7B (H=3584, V=152064) GRPO, math-shape
synthetic rollouts, G=8, 2k context — weak-scaled: 16 prompts x 8 rollouts = 128 rows (~100k response tokens) per
GPU, i.e. the reference's 128-prompt batch at 8 GPUs.  Random-init lm_head, random hidden states, random tokens
("data": "synthetic"); the transformer body is outside the measured path (SURVEY.md section 8).

One *step* = one policy update over one batch:
  device-resident (``value``):  segmented advantage kernel -> response-mask reductions (+16-byte count all-reduce)
     -> per 18944-token chunk: fused tcgen05 lm_head forward (GEMM + softmax statistics; --gemm-impl library: cuBLAS + the
        streaming logprob+loss kernel), partial merge + loss epilogue, fused backward (in place), dH and dW GEMMs
     -> gradient all-reduce (N>1; the last chunk's dW in 8 slices, each all-reduced as soon as final) -> metric sums
     -> fused clip + AdamW + bf16 cast step on the lm_head.
  end-to-end (``e2e``): the same through the public API from host objects: Episode lists -> step table -> C++
     prefix-merge packer -> pinned staging -> H2D -> [all of the above] -> D2H of the advantages (Step.advantage
     mutation) and the metric sums.  Hidden states stay on the device (they are produced there by the model body).
A token = one response-region token of a packed row (SURVEY.md section 8d).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
# stdout carries exactly one JSON line (rank 0).  Libraries (NCCL's version banner, ...) write to fd 1 as well, so
# fd 1 is pointed at stderr for the life of the process and the result goes to a private duplicate of the real stdout.
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj: dict) -> None:
    _RESULT_OUT.write(json.dumps(obj) + "\n")
    _RESULT_OUT.flush()

METRIC = "policy-update tokens/sec (GRPO, 7B, G=8, 2k ctx)"
UNIT = "tokens/s"
WORKLOAD = "qwen7b-math"
PROMPTS_PER_GPU = 16


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])), smax.append(float(parts[2])), power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None, "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference's path (oracle port) on host cores, bounded sample
# --------------------------------------------------------------------------------------------------
_CPU_CACHE: dict = {}


def _reference_host_stages(episodes, spec):
    """C1-C3 of BASELINE.md section 4 on the reference's OWN code (unmodified, located by oracle/ref_harness, which also
    stubs the third-party imports it cannot resolve here): episodes -> groups ->
    rejection filter -> numpy float64 advantages -> Python prefix-merge packing into the padded DataProto -> token-level
    advantage broadcast.  Returns (seconds, response tokens, rows as python lists for the loss sample, adv by uid)."""
    from types import SimpleNamespace

    from oracle import ref_harness as rh

    m = rh.load()
    C, TF, RS, A, VT = m["config"], m["transform"], m["rejection_sampling"], m["advantage"], m["verl_transform"]
    key = ("ref_eps", id(episodes))
    if key not in _CPU_CACHE:  # conversion into the reference's pydantic objects is input preparation (untimed)
        _CPU_CACHE.clear()
        _CPU_CACHE[key] = rh.to_reference_episodes(episodes)
    ref_eps = _CPU_CACHE[key]
    for ep in ref_eps:
        for t in ep.trajectories:
            for st in t.steps:
                st.advantage = None
    algo = C.AlgorithmConfig(estimator=C.rLLMAdvantageEstimator(spec.estimator))
    engine = SimpleNamespace(tokenizer=SimpleNamespace(pad_token_id=151643), processor=None)
    t0 = time.perf_counter()
    groups, _ = TF.transform_episodes_to_trajectory_groups(ref_eps, C.TransformConfig(), C.CompactFilteringConfig())
    f_groups, f_eps, _ = RS.apply_rejection_sampling_and_filtering(ref_eps, groups, C.RejectionSamplingConfig(mode="none", min_trajs_per_group=2), RS.RejectionSamplingState())
    batch = VT.transform_episodes_to_dataproto(f_eps, engine, spec.max_prompt_length, spec.max_prompt_length + spec.max_response_length)
    A.collect_reward_and_advantage_from_trajectory_groups(f_groups, algo)
    batch = VT.update_dataproto_with_advantages(batch, f_eps, mode="broadcast")
    t_host = time.perf_counter() - t0
    resp_mask, responses, adv = batch.batch["response_mask"], batch.batch["responses"], batch.batch["advantages"]
    att = batch.batch["attention_mask"][:, -responses.shape[1]:]
    lens = att.sum(-1)  # response-region tokens per row (mask 0 or 1)
    return t_host, int(lens.sum()), {"responses": responses, "mask": resp_mask, "adv": adv, "lens": lens}


def cpu_reference_step(episodes, spec, loss_kw, sample_tokens: int, seed: int = 0) -> dict:
    """One pass of the reference's CPU path on the same workload.  Host stages (transform, rejection filter, numpy
    advantages, Python prefix-merge packing, padded tensors, token-level advantage broadcast): the reference's own code
    when it is present (kind "reference"), else the oracle port of it (kind "port").  lm_head + verl loss
    forward/backward: restated in torch-CPU on a bounded token sample (the reference has no local loss: it lives in
    verl's workers / the remote Tinker service)."""
    from oracle import loss_oracle as lo
    from oracle import ref_harness as rh

    torch.set_num_threads(os.cpu_count() or 1)
    kind = "reference" if rh.available() else "port"
    if kind == "reference":
        t_host, n_resp, padded = _reference_host_stages(episodes, spec)
        lens_all = padded["lens"]
        take, tok = 0, 0
        while take < len(lens_all) and tok < sample_tokens:
            tok += int(lens_all[take])
            take += 1
        lens = lens_all[:take]
        sel = torch.arange(padded["responses"].shape[1])[None, :] < lens[:, None]
        labels = padded["responses"][:take][sel].long()
        mask = padded["mask"][:take][sel].to(torch.uint8)
        row_adv = torch.stack([padded["adv"][i][padded["mask"][i] != 0][:1].sum() for i in range(take)]).float()  # the row's scalar (0 for all-masked rows)
    else:
        from oracle import advantage_oracle as ao
        from oracle import pack_oracle as po

        t0 = time.perf_counter()
        from rllm_b200 import transform as tf
        from rllm_b200.config import TransformConfig

        groups, _ = tf.transform_episodes_to_trajectory_groups(episodes, TransformConfig())
        adv_by_uid, _ = ao.collect(groups, spec.estimator)
        rows = po.rows_from_episodes(episodes)
        batch = po.padded_batch(rows, 151643, spec.max_prompt_length, spec.max_prompt_length + spec.max_response_length)
        po.advantages_tensor(rows, adv_by_uid, batch["response_mask"])
        t_host = time.perf_counter() - t0
        n_resp = int(sum(min(len(r["response"]), batch["responses"].shape[1]) for r in rows))
        take, tok = 0, 0
        while take < len(rows) and tok < sample_tokens:
            tok += len(rows[take]["response"])
            take += 1
        lens = torch.tensor([len(r["response"]) for r in rows[:take]])
        labels = torch.tensor([t for r in rows[:take] for t in r["response"]], dtype=torch.long)
        mask = torch.tensor([m for r in rows[:take] for m in r["mask"]], dtype=torch.uint8)
        row_adv = torch.tensor([adv_by_uid[r["step_id"]] for r in rows[:take]], dtype=torch.float32)

    # bounded loss sample: the first rows until `sample_tokens` response tokens
    g = torch.Generator().manual_seed(seed)
    T = int(lens.sum())
    seq_id = torch.repeat_interleave(torch.arange(take), lens)
    hidden = torch.randn(T, spec.hidden, generator=g)
    if "w" not in _CPU_CACHE:  # synthetic lm_head, generated once (untimed)
        _CPU_CACHE["w"] = torch.randn(spec.vocab, spec.hidden, generator=torch.Generator().manual_seed(0)) * 0.02
    weight = _CPU_CACHE["w"].clone().requires_grad_(True)
    old = -12.0 + 0.05 * torch.randn(T, generator=g)  # ~ log(1/V) for random labels under a random-init head
    t1 = time.perf_counter()
    hid = hidden.detach().requires_grad_(True)
    logits = hid @ weight.t()  # fp32 MKL GEMM: the fastest lm_head this host can do (bf16 has no fast CPU path here)
    out = lo.policy_loss(logits, labels, mask, seq_id, row_adv, lo.LossSpec(**loss_kw), old_logp=old, dtype=torch.float32)
    out["loss"].backward()
    t_loss = time.perf_counter() - t1
    per_tok = t_host / max(n_resp, 1) + t_loss / max(T, 1)
    return {"tokens_per_s": 1.0 / per_tok, "host_s": t_host, "host_tokens": n_resp, "loss_s": t_loss, "loss_tokens": T, "loss": float(out["loss"].detach()), "kind": kind}


# --------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed, for comparing two builds output by output
# --------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 21  # elements kept of a larger output: 8 MB in float32, so the 8 outputs stay under 64 MB in all
DUMP_SEED = 0


def dump_outputs(out_dir: Path, outputs: dict) -> None:
    """Write each output as ``out_dir/<name>.npy``: float64 arrays as they are, tensors in float32 (bf16 widened).  A tensor of
    more than DUMP_SAMPLE elements is flattened and sampled at DUMP_SEED-seeded positions (sorted, drawn with replacement),
    which depend only on its size: the same arguments give the same sample in every run and in every build.  None: skipped."""
    out_dir.mkdir(parents=True, exist_ok=True)
    total = 0
    for name, t in outputs.items():
        if t is None:
            continue
        if isinstance(t, torch.Tensor):
            flat = t.detach().reshape(-1)
            if flat.numel() > DUMP_SAMPLE:
                idx = np.sort(np.random.default_rng(DUMP_SEED).integers(0, flat.numel(), DUMP_SAMPLE))
                flat = flat[torch.from_numpy(idx).to(flat.device)]
            t = flat.float().cpu().numpy()
        assert t.dtype in (np.float32, np.float64), (name, t.dtype)
        total += t.nbytes
        assert total <= 64 << 20, f"outputs past {name} exceed 64 MB"
        np.save(out_dir / f"{name}.npy", t)
    log(f"dumped {', '.join(k for k, v in outputs.items() if v is not None)} ({total / 2**20:.1f} MB) to {out_dir}")


# --------------------------------------------------------------------------------------------------
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"], help="ours; reference = the reference's CPU path; torch_gpu = stock torch / verl-style unfused update on the same GPU (comparator)")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--workload", default=WORKLOAD)
    ap.add_argument("--prompts-per-gpu", type=int, default=0, help="0 = the workload's 8-GPU batch / 8")
    ap.add_argument("--chunk-tokens", type=int, default=18944, help="tokens per lm_head chunk; 18944 = 148 x 128: the dH GEMM (14 column blocks) fills whole waves of 74 CTA pairs")
    ap.add_argument("--cpu-sample-tokens", type=int, default=3072, help="response tokens of the CPU arm's lm_head + loss sample (about 20-30 s of host work per step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gemm-impl", default=os.environ.get("RLLM_B200_GEMM_IMPL", "tcgen05"), choices=["hybrid", "tcgen05", "library"], help="lm_head GEMMs: hand-written tcgen05 CTA-pair kernels with the fused statistics epilogue, or cuBLAS + the streaming softmax/loss kernel")
    ap.add_argument("--optimizer-impl", default="fused", choices=["fused", "torch"], help="AdamW step: hand-written norm+clip+AdamW+cast+reset passes, or clip_grad_norm_ + torch.optim.AdamW(fused) + copy")
    ap.add_argument("--timeline", default="", help="write the kernel timeline of one update step per rank (CUPTI through torch.profiler, after the timed region) to <prefix>_rank<r>.json; tools/timeline_summary.py reads it")
    ap.add_argument("--dense", action="store_true", help="disable the exact token compaction (every response token through every kernel)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="after the timed update steps, write what the last one computed to DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU update step; the reference arm has none")

    from rllm_b200.synth import WORKLOADS, make_episodes

    spec = WORKLOADS[args.workload]
    if args.prompts_per_gpu <= 0:  # weak scaling of the reference batch: its global prompt count spread over 8 GPUs
        args.prompts_per_gpu = max(1, spec.prompts // 8) if spec.name != "qwen1.5b-gsm8k" else spec.prompts  # configs[1] is a 1-GPU config
    loss_kw = dict(loss_agg_mode="seq-mean-token-mean", clip_ratio_low=0.2, clip_ratio_high=0.28)  # cookbooks/math/train_verl.sh:36-39
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    config = {
        "workload": f"{spec.name}: {spec.model} lm_head tail (H={spec.hidden}, V={spec.vocab}), {spec.estimator.upper()} G={spec.group}, {spec.ctx} ctx, {args.prompts_per_gpu} prompts x {spec.group} rollouts per GPU (weak scaling of the {spec.prompts}-prompt batch: the N-GPU batch is N copies of the per-GPU draw under distinct task ids, i.e. exactly the 1-GPU work per GPU)",
        "global_batch_rows": args.prompts_per_gpu * spec.group * max(args.gpus, 1),
        "parallelism": f"dp{args.gpus}",
        "loss": "verl vanilla PPO clip 0.2/0.28 + dual-clip 3.0, seq-mean-token-mean, KL off, entropy off; pi_old = recomputed log-probs + N(0, 0.05^2) (device-resident stage-5 output)",
        "dp_balance": "shards balanced on the sweep's work (tokens with a non-zero advantage count 3x) and on each rank's measured throughput (adaptive; 5 untimed rounds after the warm-up, forward+backward and forward-only trajectories split separately)" if args.gpus > 1 else "n/a",
        "chunk_tokens": args.chunk_tokens,
        "token_compaction": "off (dense)" if args.dense else "on (exact: unmasked tokens dropped; zero-advantage tokens forward-only)",
        "gemm_impl": args.gemm_impl, "optimizer_impl": args.optimizer_impl,
        "cache": "inputs larger than L2 (5 GB logits chunk, 1.1 GB lm_head, 0.7 GB hidden states)",
    }

    # ---------------- reference (CPU) arm ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        episodes = make_episodes(spec, seed=0, prompts=args.prompts_per_gpu, replicas=max(args.gpus, 1))
        for _ in range(args.warmup):
            cpu_reference_step(episodes, spec, loss_kw, 64)
        vals = [cpu_reference_step(episodes, spec, loss_kw, args.cpu_sample_tokens, seed=i) for i in range(args.steps)]
        v = float(np.median([x["tokens_per_s"] for x in vals]))
        src = "the reference's own code (unmodified, third-party imports stubbed)" if vals[0]["kind"] == "reference" else "the oracle port of the reference's code"
        sample = f"per step: transform + rejection filter + numpy advantages + Python prefix-merge packing + padded tensors + advantage broadcast by {src} on all {vals[0]['host_tokens']} response tokens ({vals[0]['host_s']*1e3:.0f} ms); lm_head + verl loss fwd/bwd restated in torch CPU (fp32 GEMM, all cores; the reference has no local loss) on the first {vals[0]['loss_tokens']} tokens ({vals[0]['loss_s']:.1f} s), per-token rates combined"
        emit({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(np.median([x["host_s"] + x["loss_s"] for x in vals])), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": vals[0]["kind"], "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        })
        return

    # ---------------- our arm ----------------
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device"
    from rllm_b200 import loss as L
    from rllm_b200 import transform as tf
    from rllm_b200.backend import PolicyUpdateEngine, SyntheticPolicyHead
    from rllm_b200.config import AlgorithmConfig, PolicyLossConfig, TransformConfig
    from rllm_b200.dp import DPContext

    dp = DPContext.from_env()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    assert dp.world_size == max(args.gpus, 1), f"--gpus {args.gpus} but WORLD_SIZE={dp.world_size} (launch N>1 under torchrun)"

    # same on every rank; N GPUs: N copies of the per-GPU draw under distinct task ids, so the work per GPU is exactly the
    # 1-GPU run's at every N (weak scaling without the sample-to-sample variation of lengths / uniform groups)
    episodes = make_episodes(spec, seed=0, prompts=args.prompts_per_gpu, replicas=dp.world_size)
    groups, _ = tf.transform_episodes_to_trajectory_groups(episodes, TransformConfig())
    cfg = PolicyLossConfig(**loss_kw)
    algo = AlgorithmConfig(estimator=spec.estimator)
    policy = SyntheticPolicyHead(spec.vocab, spec.hidden, dev, seed=0)
    eng = PolicyUpdateEngine(policy, cfg, algo, dp=dp, chunk_tokens=args.chunk_tokens, max_response_length=spec.max_prompt_length + spec.max_response_length, compact_tokens=not args.dense, gemm_impl=args.gemm_impl, optimizer_impl=args.optimizer_impl)

    g = torch.Generator(device=dev).manual_seed(1234 + rank)

    def prepare():
        """Pack this rank's shard (DP: balanced on the sweep's work — active tokens count 3x — and, once sweeps have been timed,
        on each rank's measured throughput), H2D, hidden states, and stage 5 once, untimed: pi_old log-probs of the current
        weights (device-resident afterwards), made slightly off-policy (sigma 0.05) so that the clip branches are exercised."""
        pb_ = eng.pack(episodes=episodes, groups=groups, sharded=True)
        db_ = eng.shard_to_device(pb_)
        hidden_ = policy.hidden_states(pb_, db_)
        eng.old_log_probs(pb_, db_, hidden_)
        db_.old_logp = db_.old_logp + 0.05 * torch.randn(db_.n_tokens, generator=g, device=dev)
        return pb_, db_, hidden_

    pb, db, hidden = prepare()
    tok_t = torch.tensor([pb.n_tokens], dtype=torch.int64, device=dev)
    dp.all_reduce_sum_(tok_t)
    global_tokens = int(tok_t.item())
    log(f"[rank {rank}] rows={db.n_rows} tokens={db.n_tokens} global_tokens={global_tokens} pack={eng.timings.pack_s*1e3:.1f} ms")

    def phase(name, fn):  # CUDA-event bracket of a step phase that is not one of the lm_head sweep's kernels
        pe = eng.head.profile_events
        if pe is None:
            return fn()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        r = fn()
        eb.record()
        pe.append((name, 0, ea, eb))
        return r

    last_step = {}  # what the last device step returned beyond the metric sums (kept for --dump-outputs only)

    def device_step():
        phase("advantages+weights", lambda: (eng.advantages(pb, db, groups), eng.loss_weights(db)))
        res = eng.forward_backward(pb, db, hidden)
        phase("grad_allreduce_exposed", eng.reduce_gradients)  # the part of the all-reduce not hidden under the last dH GEMM
        sums = phase("metric_sums", eng.reduce_metrics)
        grad_norm = phase("optimizer", eng.optimizer_step)
        if args.dump_outputs:
            last_step.update(res=res, grad_norm=grad_norm)
        return sums

    def e2e_step():
        pb2 = eng.pack(episodes=episodes, groups=groups, sharded=True)  # host: this rank's share -> step table -> C++ prefix-merge into pinned staging
        db2 = eng.shard_to_device(pb2)  # H2D
        db2.old_logp = db.old_logp  # stage-5 outputs, produced on the device (log-probs and the softmax reference point)
        db2.lse_ref = db.lse_ref
        eng.advantages(pb2, db2, groups)  # includes the D2H of the advantages for Step.advantage
        eng.loss_weights(db2)
        eng.forward_backward(pb2, db2, hidden)
        eng.reduce_gradients()
        sums = eng.reduce_metrics()  # D2H of the metric sums
        eng.optimizer_step()
        return sums, db2

    def timed(fn, steps, profile=False):
        dp.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eng.head.profile_events = [] if profile else None
        eng.timings.launches = 0
        t0 = time.perf_counter()
        a.record()
        last = None
        for _ in range(steps):
            last = fn()
        b.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dp.barrier()
        ms = torch.tensor([a.elapsed_time(b), wall * 1e3], dtype=torch.float64, device=dev)
        dp.all_reduce_max_(ms)
        ev = eng.head.profile_events
        eng.head.profile_events = None
        return float(ms[0]), float(ms[1]), last, ev

    for _ in range(args.warmup):
        device_step()
    if dp.enabled and eng.adaptive_balance:
        # what a training loop gets from its second step on: the partition follows the ranks' measured sweep throughput
        # (GPUs of one box differ by a few % under the power cap, and the closed-loop trim needs a few steps to settle).
        # Five rounds of re-partition + one step, untimed.
        for _ in range(5):
            pb, db, hidden = prepare()
            if rank == 0:
                log(f"[rank 0] balance round: speeds={None if eng.rank_speeds is None else np.round(eng.rank_speeds, 4).tolist()} {eng.last_balance}")
            device_step()
        eng.adaptive_balance = False  # freeze the estimate: every later pack of the run (e2e steps) reproduces this partition
        log(f"[rank {rank}] rebalanced: tokens={db.n_tokens} rank_speeds={None if eng.rank_speeds is None else np.round(eng.rank_speeds, 4).tolist()}")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dev_ms, _, sums, events = timed(device_step, args.steps, profile=True)
    if args.dump_outputs and rank == 0:
        res = last_step["res"]
        master = eng._master if eng._master is not None and eng._master.shape == policy.weight.shape else None  # None: sharded (ZeRO-1)
        dump_outputs(Path(args.dump_outputs), {
            "advantages": db.row_adv, "logp": res.logp, "entropy": res.entropy, "d_hidden": res.d_hidden,
            "metric_sums": np.array([sums[k] for k in L.N.SUM_NAMES], dtype=np.float64), "grad_norm": np.array([last_step["grad_norm"]], dtype=np.float64),
            "lm_head_weight": policy.weight, "lm_head_master": master,
        })
    launches_per_step = eng.timings.launches / args.steps + 3  # + the three advantage kernels
    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    _, e2e_wall_ms, (e2e_sums, db2), _ = timed(e2e_step, args.steps)
    clocks = sampler.stop() if rank == 0 else {}

    # stage 5 alone (old / ref log-prob pass: lm_head GEMM + fused forward in no-loss mode), reported beside the step
    def stage5():
        eng.wait_weights()
        eng.head.logprobs(hidden, policy.weight, db, cfg)

    stage5()
    s5_ms, _, _, _ = timed(stage5, args.steps)

    # stage 5 + update as ONE step (what a trainer step pays around the policy update): pi_old pass with the current
    # weights, then the update.  "reuse": the pass keeps the logits of the tokens the update back-propagates and the update
    # runs no lm_head forward (weights unchanged in between — the reference's default of one epoch / one mini-batch);
    # "recompute": the round-1 composition (statistics-only pass, the update recomputes its forward).
    noise = 0.05 * torch.randn(db.n_tokens, generator=g, device=dev)

    def full_step(reuse: bool):
        eng.reuse_forward = reuse
        eng.old_log_probs(pb, db, hidden, groups=groups if reuse else None)
        db.old_logp = db.old_logp + noise  # synthetic off-policy-ness so that the clip branches are exercised
        return device_step()

    full = {}
    for name, reuse in (("recompute", False), ("reuse", True)):
        for _ in range(2):
            full_step(reuse)
        ms, _, fsums, fev = timed(lambda: full_step(reuse), args.steps, profile=True)
        shares = {}
        for nm, n, ea, eb in fev:
            shares[nm] = shares.get(nm, 0.0) + ea.elapsed_time(eb)
        full[name] = {"tokens_per_s": global_tokens * args.steps / (ms / 1e3), "ms_per_step": ms / args.steps, "loss": fsums["loss"], "ms_per_step_by_op": {k: round(v / args.steps, 3) for k, v in shares.items()},
                      "compaction": dict(eng.last_compaction)}
    eng.reuse_forward = True
    value = global_tokens * args.steps / (dev_ms / 1e3)
    e2e_value = global_tokens * args.steps / (e2e_wall_ms / 1e3)

    # per-kernel shares from the CUDA events recorded inside the timed region
    per = {}
    for name, n, ea, eb in events:
        d = per.setdefault(name, {"ms": 0.0, "tokens": 0, "launches": 0})
        d["ms"] += ea.elapsed_time(eb)
        d["tokens"] += n
        d["launches"] += 1
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    V, H = spec.vocab, spec.hidden
    alg = {  # algorithmic work per token (DESIGN.md section 4)
        "loss_fwd": ("hbm", V * 2 + 40), "loss_bwd": ("hbm", 2 * V * 2),
        "gemm_fwd": ("tensor", 2 * H * V), "gemm_dh": ("tensor", 2 * H * V), "gemm_dw": ("tensor", 2 * H * V),
        "gemm_fwd_stats": ("tensor", 2 * H * V), "loss_merge": ("hbm", 16 * ((V + 255) // 256) + 40),
    }
    kernels, phases = {}, {}
    for name, d in per.items():
        if name not in alg:
            phases[name] = {"ms_per_step": d["ms"] / args.steps, "share_of_step": d["ms"] / dev_ms}
            continue
        bound, work = alg[name]
        rate = work * d["tokens"] / (d["ms"] / 1e3)
        peak = hbm_peak * 1e9 if bound == "hbm" else tf_peak * 1e12
        kernels[name] = {"bound": bound, "share_of_step": d["ms"] / dev_ms, "ms_per_launch": d["ms"] / d["launches"], "achieved": rate / (1e9 if bound == "hbm" else 1e12), "unit": "GB/s" if bound == "hbm" else "TFLOP/s", "frac": rate / peak}
    fwd = kernels.get("loss_fwd", {})
    traffic, traffic_src = None, None
    try:  # DRAM bytes per launch from the committed `ncu --set full` capture of this command (full 16384-token chunk)
        cap = json.loads((ROOT / "profiles" / "r01_ncu_bench_loss_traffic.json").read_text())
        k = next(v for name, v in cap.items() if "loss_fwd_stream" in name)
        traffic = float(np.mean([x["dram_read_bytes"] + x["dram_write_bytes"] for x in k]))
        traffic_src = "profiles/r01_ncu_bench_loss_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per 16384-token launch; algorithmic bytes of that launch: %d)" % (16384 * (V * 2 + 40))
    except Exception:
        pass
    if args.gemm_impl in ("tcgen05", "hybrid"):
        # dominant kernel by time: the fused lm_head forward (tcgen05 GEMM + softmax-statistics epilogue); tensor bound
        gf = kernels.get("gemm_fwd_stats", {})
        gtraffic, gsrc = None, None
        try:  # DRAM bytes per launch from the committed `ncu --set full` capture of this command (one full chunk)
            cap = json.loads((ROOT / "profiles" / "r02_ncu_kernels.json").read_text())
            name = next(n for n in cap["kernels"] if "pair_gemm_kernel<0, 0, 1" in n)
            gtraffic = float(np.mean([x["dram_read_bytes"] + x["dram_write_bytes"] for x in cap["kernels"][name]]))
            gsrc = cap.get("source", "") + f"; dram__bytes_read.sum + dram__bytes_write.sum per {args.chunk_tokens}-token launch (logits written: {args.chunk_tokens * V * 2} B of it)"
        except Exception:
            pass
        roofline = {
            "kernel": "pair_gemm_kernel<K-major, K-major, bf16 store + softmax statistics> (tcgen05 cta_group::2 lm_head forward fused with log-softmax / entropy statistics)",
            "bound": "tensor", "achieved": gf.get("achieved"), "peak": tf_peak, "unit": "TFLOP/s", "frac": gf.get("frac"), "traffic": gtraffic, "traffic_source": gsrc,
            "peak_source": peak_src + " bf16_tflops_sustained (kernel timed inside a long step)", "algorithmic_flops_per_token": 2 * H * V, "share_of_step": gf.get("share_of_step"),
            "note": ("all three lm_head GEMMs are the hand-written tcgen05 kernel" if args.gemm_impl == "tcgen05" else "forward = hand-written tcgen05 kernel, dH / dW = library GEMMs (cuBLAS)") + "; `kernels` lists every op's share and fraction; with the entropy term off the forward stores E = exp(z - lse_old) and there is no d-logits pass (DESIGN 4e; loss_bwd_stream_kernel otherwise)",
        }
    else:
        roofline = {
            "kernel": "loss_fwd_stream_kernel (fused log-softmax + gather + entropy + PPO loss forward; the kernel north_star names)",
            "bound": "hbm", "achieved": fwd.get("achieved"), "peak": hbm_peak, "unit": "GB/s", "frac": fwd.get("frac"), "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "algorithmic_bytes_per_token": V * 2 + 40, "share_of_step": fwd.get("share_of_step"),
            "note": "the lm_head GEMMs (cuBLAS, library) dominate the step by time; see `kernels` for every op's share and fraction",
        }

    # GPU comparator: the same update as stock torch / verl-style unfused ops would run it on this GPU (tools/comparators.py)
    if args.timeline:  # evidence for the overlap of the gradient exchange with the GEMMs: which kernels ran when, on which stream
        try:
            import tempfile
            from torch.profiler import ProfilerActivity, profile

            dp.barrier()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                device_step()
                torch.cuda.synchronize()
            with tempfile.NamedTemporaryFile(suffix=".json") as tf_:
                prof.export_chrome_trace(tf_.name)
                trace = json.load(open(tf_.name))
            evs = [e for e in trace.get("traceEvents", []) if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset") and "ts" in e]
            t0 = min(e["ts"] for e in evs)
            rows = [{"name": e["name"][:96], "cat": e["cat"], "start_us": round(e["ts"] - t0, 1), "dur_us": round(e.get("dur", 0.0), 1), "stream": e.get("args", {}).get("stream")} for e in sorted(evs, key=lambda e: e["ts"])]
            json.dump({"rank": rank, "world_size": dp.world_size, "kernels": rows}, open(f"{args.timeline}_rank{rank}.json", "w"))
        except Exception as e:  # the timeline is evidence, not part of the measurement
            log(f"[rank {rank}] timeline unavailable: {type(e).__name__}: {e}")

    gpu_baseline = None
    if dp.world_size == 1 and (not args.no_gpu_baseline or args.impl == "torch_gpu"):
        sys.path.insert(0, str(ROOT / "tools"))
        from comparators import TorchGpuUpdate

        del eng.head._resident_logits, eng.head._logits  # give the comparator the memory
        eng.head._resident_logits = eng.head._logits = None
        torch.cuda.empty_cache()
        cmp_ = TorchGpuUpdate(policy.weight, loss_agg_mode=cfg.loss_agg_mode, clip_low=cfg.clip_ratio_low, clip_high=cfg.clip_ratio_high, clip_c=cfg.clip_ratio_c)
        seq_t = torch.from_numpy(pb.seq_ids()).to(dev).long()
        lab_t, msk_t = db.labels.long(), db.mask.bool()

        def torch_step():
            return cmp_.step(hidden, lab_t, msk_t, seq_t, db.row_adv, db.old_logp)

        for _ in range(2):
            torch_step()
        tg_ms, _, tg_out, _ = timed(torch_step, args.steps)
        gpu_baseline = {
            "value": global_tokens * args.steps / (tg_ms / 1e3), "unit": UNIT, "ms_per_step": tg_ms / args.steps, "loss_last_step": float(tg_out["loss"]),
            "what": "stock torch on the same GPU, nothing of this repo: per <=16384-token micro-batch torch.matmul lm_head -> [n,V] logits -> logprobs_from_logits (" + ("flash-attn Triton cross-entropy" if cmp_.ce is not None else "fp32 logsumexp + gather") + ") -> vanilla PPO clip/dual-clip, seq-mean-token-mean -> autograd backward (bf16 dH/dW) -> clip_grad_norm_ + torch.optim.AdamW(fused) on an fp32 master + bf16 cast; every response token (no compaction)",
            "ours_over_torch": value / (global_tokens * args.steps / (tg_ms / 1e3)),
        }
        del cmp_
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and dp.world_size == 1 and not args.no_cpu_baseline and args.impl != "torch_gpu":
        cpu = cpu_reference_step(episodes, spec, loss_kw, args.cpu_sample_tokens)
        cpu_baseline = {
            "value": cpu["tokens_per_s"], "unit": UNIT, "cores": cores, "kind": cpu["kind"],
            "sample": f"{'the reference itself' if cpu['kind'] == 'reference' else 'oracle port of the reference'}: transform + filter + advantages + Python prefix-merge packing + padded tensors on all {cpu['host_tokens']} tokens ({cpu['host_s']*1e3:.0f} ms); lm_head + verl loss fwd/bwd restated in torch-CPU on {cpu['loss_tokens']} tokens ({cpu['loss_s']:.1f} s), per-token rates combined",
        }

    if rank == 0 and args.impl == "torch_gpu" and gpu_baseline is None:
        emit({"impl": "torch_gpu", "unavailable": "the stock-torch comparator is a single-GPU arm (run it with --gpus 1)"})
    elif rank == 0 and args.impl == "torch_gpu":
        emit({"impl": "torch_gpu", "metric": METRIC, "value": gpu_baseline["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": gpu_baseline["ms_per_step"],
              "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": dict(config, gemm_impl="cuBLAS (torch.matmul)", token_compaction="off"),
              "gpu_baseline": gpu_baseline, "clocks": clocks})
    elif rank == 0:
        emit({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": dp.world_size, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_wall_ms / args.steps, "h2d_bytes_per_step": int(eng.timings.h2d_bytes + 8 * len(groups) * spec.group), "d2h_bytes_per_step": int(eng.timings.d2h_bytes + 8 * len(groups) * spec.group + 16), "host_pack_ms": eng.timings.pack_s * 1e3},
            "gpu_launches": int(round(launches_per_step * args.steps)),
            "roofline": roofline, "kernels": kernels, "phases": phases, "cpu_baseline": cpu_baseline, "gpu_baseline": gpu_baseline, "clocks": clocks,
            "value_with_stage5": {"value": full["reuse"]["tokens_per_s"], "unit": UNIT, "reuse": full["reuse"], "recompute": full["recompute"],
                                  "note": "pi_old log-prob pass + policy update timed as one step (CUDA events, same barriers as `value`). `value` itself stays the update alone with its forward recomputed, as in round 1; with the forward reused the update alone would be faster still but its forward lives in the pi_old pass, so only this combined number is quoted for it"},
            "stage5_logprob_pass": {"tokens_per_s": global_tokens * args.steps / (s5_ms / 1e3), "ms": s5_ms / args.steps, "note": "pi_old / reference-policy log-prob + entropy pass over all response tokens (not part of `value`)"},
            "loss": sums["loss"], "masked_tokens_per_step": sums["mask"], "tokens_per_step": global_tokens,
            "compaction": dict(eng.last_compaction, note="rank-0 shard; exact elimination of unmasked tokens and of the backward of zero-advantage tokens (DESIGN.md section 4b)") if eng.compact_tokens else None,
        })
    if dp.enabled:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
