"""bench.py's extra measurements after the timed region (reconfiguration after a kill, BASELINE config 4 at N = 8) must
never cost the throughput line: every run is bounded, all of them share one budget (the driver allows a bench.py run
870 s), failures are reported inside the JSON.  The subprocesses need GPUs; here they are replaced by fakes and only the
host logic around them runs."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


class FakePopen:
    """Stands in for subprocess.Popen: ``script`` maps a predicate on the command line to (stdout, returncode) or to
    the string "hang" (communicate raises TimeoutExpired)."""
    script = []
    commands = []

    def __init__(self, cmd, **kw):
        self.cmd, self.pid, self.returncode = cmd, 2 ** 22 + 12345, 0       # a pid nobody owns: killpg raises, is caught
        FakePopen.commands.append(cmd)
        assert kw.get("start_new_session") is True                          # the whole process group can be killed
        assert "RANK" not in kw["env"] and "MASTER_PORT" not in kw["env"]   # nothing of the outer torchrun leaks in
        self.behaviour = next(b for pred, b in FakePopen.script if pred(cmd))

    def communicate(self, timeout=None):
        assert timeout is not None and timeout > 0
        self.timeout = timeout
        if self.behaviour == "hang":
            raise subprocess.TimeoutExpired(self.cmd, timeout)
        out, self.returncode = self.behaviour
        return out, ""

    def wait(self):
        return -9


def reconfig_line(value, replicas, stages):
    return json.dumps({"metric": "reconfiguration_latency_s", "value": value,
                       "config": {"workload": f"gpt2-xl: {replicas} replicas x {stages} stages"},
                       "pipelines_after": [[4, 5, 6], [0, 1, 2, 3]],
                       "notify_to_pipelines_rebuilt_and_states_copied_s": value / 2,
                       "replicas_identical_after": True, "tokens_per_step": 131072,
                       "step_s_before": {"median": 0.8, "max": 0.81, "n": 3},
                       "step_s_after": {"median": 1.0, "max": 1.1, "n": 3}})


def install(monkeypatch, script):
    FakePopen.script, FakePopen.commands = script, []
    monkeypatch.setattr(subprocess, "Popen", FakePopen)
    monkeypatch.setenv("RANK", "0")
    monkeypatch.setenv("MASTER_PORT", "29500")


def test_reconfiguration_record_from_both_runs(monkeypatch):
    install(monkeypatch, [(lambda c: c[c.index("--replicas") + 1] == "2", ("noise\n" + reconfig_line(3.5, 2, 4) + "\n", 0)),
                          (lambda c: c[c.index("--replicas") + 1] == "1", (reconfig_line(4.25, 1, 8) + "\n", 0))])
    out = bench.embedded_reconfiguration("gpt2-xl", 8, time.perf_counter() + 400)
    assert out["two_replicas"]["value"] == 3.5 and out["lone_pipeline"]["value"] == 4.25
    assert out["value"] == 4.25                                   # the worse of the two is the headline latency
    assert out["two_replicas"]["tokens_per_s_before"] == 131072 / 0.8      # config 4's shape at N = 8: 2 x 4 stages
    assert out["two_replicas"]["tokens_per_s_after"] == 131072 / 1.0       # 4 + 3 stages
    assert [c[c.index("--gpus") + 1] for c in FakePopen.commands] == ["8", "8"]
    assert out["higher_is_better"] is False and out["unit"] == "s"


def test_a_hanging_run_is_killed_and_reported_and_the_next_is_not_started(monkeypatch):
    install(monkeypatch, [(lambda c: True, "hang")])
    out = bench.embedded_reconfiguration("gpt2-xl", 8, time.perf_counter() + 400)
    assert "exceeded" in out["two_replicas"]["error"]
    assert "lone_pipeline" not in out and len(FakePopen.commands) == 1
    assert out["value"] is None


def test_failed_run_is_reported_and_the_other_still_measured(monkeypatch):
    install(monkeypatch, [(lambda c: c[c.index("--replicas") + 1] == "2", ("Traceback ...\n", 1)),
                          (lambda c: True, (reconfig_line(4.0, 1, 8), 0))])
    out = bench.embedded_reconfiguration("gpt2-xl", 8, time.perf_counter() + 400)
    assert out["two_replicas"] == {"error": "no result (exit code 1)"}
    assert out["lone_pipeline"]["value"] == 4.0 and out["value"] == 4.0


def test_runs_that_no_longer_fit_the_common_budget_are_skipped(monkeypatch):
    install(monkeypatch, [(lambda c: True, (reconfig_line(3.0, 2, 4), 0))])
    out = bench.embedded_reconfiguration("gpt2-xl", 8, time.perf_counter() + 10)
    assert "skipped" in out["two_replicas"] and "skipped" in out["lone_pipeline"] and not FakePopen.commands
    assert "skipped" in bench.embedded_config4(8, time.perf_counter() + 10)
    # a run's own bound is cut by what is left of the common budget
    out = bench.embedded_reconfiguration("gpt2-xl", 8, time.perf_counter() + 60)
    assert out["two_replicas"]["value"] == 3.0
    assert bench._run_budget(time.perf_counter() + 60) <= 60 < bench.RECONFIG_BUDGET_S
    assert bench.RECONFIG_BUDGET_S * 3 > bench.EXTRAS_BUDGET_S > bench.RECONFIG_BUDGET_S     # the cap is what binds
    assert bench.EXTRAS_BUDGET_S + 300 < 870          # headline run + parity check + extras stay inside the driver's limit


def test_lone_pipeline_needs_three_gpus(monkeypatch):
    install(monkeypatch, [(lambda c: True, (reconfig_line(1.0, 2, 1), 0))])
    out = bench.embedded_reconfiguration("gpt2", 2, None)
    assert "two_replicas" in out and "lone_pipeline" not in out


def test_config4_line_is_condensed(monkeypatch):
    line = json.dumps({"metric": "training_tokens_per_s", "value": 1.7e6, "unit": "tokens/s", "n_gpus": 8, "steps": 3,
                       "warmup": 3, "ms_per_step": 77.0, "scaling": "strong",
                       "config": {"workload": "gpt2 ...", "parallelism": "dp2 x pp4"},
                       "parity_check": {"ok": True, "loss_rel_err": 9e-8}, "stage_busy_ms": [1] * 8, "bubble_ms": [0] * 8,
                       "gpu_launches": 1234, "e2e": {"value": 1.8e6}, "engine": {"stage_layers": [5, 4, 4, 1]},
                       "roofline": {"frac": 0.1}})
    install(monkeypatch, [(lambda c: True, ("NCCL banner\n" + line + "\n", 0))])
    out = bench.embedded_config4(8, time.perf_counter() + 400)
    cmd = FakePopen.commands[0]
    assert cmd[1:3] == ["-m", "torch.distributed.run"] and "--nproc-per-node=8" in cmd
    assert cmd[cmd.index("--replicas") + 1] == "2" and cmd[cmd.index("--model") + 1] == "gpt2"
    assert cmd[cmd.index("--with-reconfig") + 1] == "0"           # the embedded run never embeds another one
    assert out["value"] == 1.7e6 and out["config"]["parallelism"] == "dp2 x pp4" and out["parity_check"]["ok"]
    assert out["stage_layers"] == [5, 4, 4, 1] and "roofline" not in out and out["wall_s"] >= 0


def test_dump_outputs_writes_the_same_sample_of_every_layer(tmp_path):
    import types

    import numpy as np
    import torch

    def layer(lid, n):
        return types.SimpleNamespace(layer_id=lid, flat_param=torch.arange(n, dtype=torch.float32) * (lid + 1))

    def engine(pipeline_id, layers):
        execution = types.SimpleNamespace(_layers=layers, total_loss=torch.tensor(3.25))
        return types.SimpleNamespace(_pipeline=types.SimpleNamespace(_pipeline_id=pipeline_id, execution=execution,
                                                                     is_last_stage=lambda: True))

    big = bench.DUMP_SAMPLE * 3
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), engine(0, [layer(0, 100), layer(7, big)]))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["layer000_param.npy", "layer007_param.npy", "total_loss.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
    assert np.load(tmp_path / "a" / "total_loss.npy") == 3.25
    assert np.array_equal(np.load(tmp_path / "a" / "layer000_param.npy"), np.arange(100, dtype=np.float32))
    sample = np.load(tmp_path / "a" / "layer007_param.npy")
    assert sample.shape == (bench.DUMP_SAMPLE,) and len(np.unique(sample)) == bench.DUMP_SAMPLE
    assert np.all(sample[1:] > sample[:-1]) and np.all(sample % 8 == 0)    # sorted positions of layer 7's values
    bench.dump_outputs(str(tmp_path / "c"), engine(1, [layer(0, 100)]))    # a second replica holds the same layers
    assert not (tmp_path / "c").exists()
