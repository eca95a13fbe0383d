"""bench.py's line assembly and teardown, exercised on the host with the device work stubbed out (no GPU, no NCCL): the JSON
line carries every key of the driver's contract at N = 1 and under a faked 2-rank launch, the phases after the timed
measurement are ordered as the multi-rank guard expects, a phase that never returns still yields the measured line on rank 0,
and `--impl reference` prints the CPU arm's line from rank 0 only.  The measurements themselves are `-m gpu` material."""
import json
import os
import sys
import tempfile
import time
import types

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import bench  # noqa: E402

CONTRACT_KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                 "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"]


class FakeEngine(object):
    def forward_backward_flops(self, batch):
        return 41.6e9 * batch

    def launches(self, training):
        return 183


class FakeRun(object):
    """Stands in for bench.TrainingRun: same attributes and return shapes, no device."""
    made = []

    def __init__(self, preset, local_batch, global_batch, rank, world, dev, dist, overlap=True, seed=1337):
        self.preset, self.B, self.global_batch, self.rank, self.world = preset, local_batch, global_batch, rank, world
        import Config
        self.cfg = Config.build_config([preset], experiment_id=0)["model_config"]
        self.t_in, self.t_out = 147443, 16389
        self.eng = FakeEngine()
        self.graph, self.graph_error = object(), None
        self.ar = types.SimpleNamespace(views=[0, 1, 2, 3]) if (world > 1 and overlap) else None
        import torch
        g = torch.Generator().manual_seed(seed)
        self.sep = types.SimpleNamespace(_loss=torch.tensor([0.07]), **{k: torch.randn(1000, generator=g)
                                                                       for k in ("params", "grads", "adam_m", "adam_v")})
        self.calls = []
        FakeRun.made.append(self)

    def prepare(self, use_graph=True):
        return use_graph

    def save_state(self):
        self.calls.append("save_state")
        return "state%d" % self.calls.count("save_state")

    def load_state(self, state, step=False):
        self.calls.append(("load_state", state, step))

    def time_steps(self, steps, warmup, prewarm_s=0.0):
        self.calls.append(("time_steps", steps))
        t = time.perf_counter()
        return 4.8 * steps, t, t + 4.8e-3 * steps

    def frames_per_step(self):
        return self.global_batch * 16389

    def e2e(self, steps, warmup):
        return {"sequential_s": 5.2e-3 * steps, "prefetch_s": 5.0e-3 * steps, "prefetch_error": None, "last_loss": 0.07,
                "bytes_h2d": 1000}


def fake_layer_table(run, iters=6):
    rows = [{"layer": "down1", "pass": p, "us": u, "gflop": 20.0, "tflops": 20.0 / u * 1e3} for p, u in (("fwd", 100.0), ("dgrad", 150.0), ("wgrad", 200.0))]
    fam = {"conv_fwd": {"us": 100.0, "gflop": 20.0, "launch_groups": 1, "tflops": 200.0},
           "conv_dgrad": {"us": 150.0, "gflop": 20.0, "launch_groups": 1, "tflops": 133.0},
           "wgrad": {"us": 200.0, "gflop": 20.0, "launch_groups": 1, "tflops": 100.0},
           "first_layer": {"us": 230.0, "gflop": 3.7, "launch_groups": 2, "tflops": 16.0}}
    return rows, fam


class Exited(Exception):
    pass


@pytest.fixture
def stubbed(monkeypatch, tmp_path):
    import torch
    import torch.distributed as dist
    FakeRun.made = []
    monkeypatch.setattr(tempfile, "tempdir", str(tmp_path))
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "empty_cache", lambda: None)
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: None)
    monkeypatch.setattr(dist, "barrier", lambda *a, **k: None)
    monkeypatch.setattr(dist, "destroy_process_group", lambda *a, **k: None)
    monkeypatch.setattr(bench, "TrainingRun", FakeRun)
    monkeypatch.setattr(bench, "layer_table", fake_layer_table)
    monkeypatch.setattr(bench, "dp_check", lambda run: {"ok": True, "replicas_identical_after_adam": True})
    monkeypatch.setattr(bench, "predict_bench", lambda rank, world, dev, dist, reps=2: {"seconds": 0.13, "n_gpus": world})
    monkeypatch.setattr(bench, "cpu_step_rate", lambda cfg, budget, steps=None, warmup=1: {
        "value": 6e4, "ms_per_step": 270.0, "steps": steps or 40, "cores": 16, "host_logical_cpus": 128, "host_physical_cores": 64,
        "sample": "stub"})

    def fake_exit(code):
        raise Exited(code)
    monkeypatch.setattr(os, "_exit", fake_exit)
    return monkeypatch


def _args(**kw):
    d = dict(gpus=1, steps=20, warmup=5, impl="ours", no_graph=False, no_overlap=False, no_extras=False, no_cpu_baseline=False,
             no_prewarm=False, dump_outputs=None)
    d.update(kw)
    return types.SimpleNamespace(**d)


def _lines(capsys):
    return [json.loads(ln) for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]


def test_single_gpu_line_has_the_contract_keys(stubbed, capsys, tmp_path, monkeypatch):
    repo, tmp = tmp_path / "repo", tmp_path / "tmp"
    repo.mkdir()
    tmp.mkdir()
    monkeypatch.setattr(bench, "REPO", str(repo))
    monkeypatch.setattr(tempfile, "tempdir", str(tmp))          # the per-layer table goes to the temporary directory
    monkeypatch.setattr(bench, "kernel_source_hash", lambda: "0" * 16)
    bench.run_ours(_args(), 0, 1, 0)
    (line,) = _lines(capsys)
    for k in CONTRACT_KEYS + ["cpu_baseline", "step_roofline", "families", "extra_configs"]:
        assert k in line, k
    assert line["n_gpus"] == 1 and line["steps"] == 20 and line["warmup"] == 5 and line["higher_is_better"] is True
    assert abs(line["ms_per_step"] - 4.8) < 1e-9
    assert abs(line["value"] - 16 * 16389 / 4.8e-3) < 1e-3
    assert abs(line["input_frames_per_s"] - 16 * 147443 / 4.8e-3) < 1e-3
    assert line["e2e"]["h2d_bytes_per_step"] == 1000 and line["e2e"]["d2h_bytes_per_step"] == 4
    assert line["e2e"]["value"] < line["value"]                 # host copies inside the timed region
    assert line["gpu_launches"] == (183 + 2) * 20
    sr = line["stack_roofline"]                                 # host-side accounting on a real engine handle (dry run)
    assert "error" not in sr and abs(sr["gflop"] - 666.0) < 0.5 and sr["passes"] == 76
    assert abs(sr["frac"] - sr["bound_ms"] / 4.8) < 1e-12 and sr["bound_ms"] < sr["bound_ms_3mma"] < 3 * sr["bound_ms"]
    assert line["roofline"]["bound"] == "tensor" and "wgrad" in line["roofline"]["kernel"]      # the time-dominant family, not the best one
    assert abs(line["roofline"]["frac"] - line["roofline"]["achieved"] / line["roofline"]["peak"]) < 1e-12
    assert line["roofline"]["traffic"] is None and "no ncu capture" in line["roofline"]["traffic_note"]
    assert set(line["extra_configs"]) == {"m6_full_multi_instrument_b32", "m5_full_learned_b16", "predict_3min_44k"}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 16
    assert "aborted_in" not in line and "dp_check" not in line
    assert FakeRun.made[0].calls == [("time_steps", 20)]
    assert os.path.exists(os.path.join(str(tmp), "wun_bench_layer_table_n1.json"))
    assert os.listdir(str(repo)) == []                          # nothing written into the tree


def test_dump_outputs_writes_a_step_from_the_seeded_start_reproducibly(stubbed, capsys, tmp_path, monkeypatch):
    """--dump-outputs DIR: after the --steps timed steps, one more step runs from the saved starting state.  Its loss, and the
    same seeded sample of its gradients, parameters and Adam slots, are written as float32 .npy files.  They are identical from
    run to run and stay within 64 MB at the benchmark's 10.3 M parameters."""
    import numpy as np
    assert 4 * 4 * bench.DUMP_SAMPLE + 4 <= 64e6
    monkeypatch.setattr(bench, "REPO", str(tmp_path))
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 300)
    dumps = []
    for k in range(2):
        d = tmp_path / ("out%d" % k)
        bench.run_ours(_args(steps=7, dump_outputs=str(d), no_extras=True, no_cpu_baseline=True), 0, 1, 0)
        (line,) = _lines(capsys)
        assert line["steps"] == 7
        # the step from the starting state, then back to the state the timed steps left for the phases that follow
        assert FakeRun.made[-1].calls == ["save_state", ("time_steps", 7), "save_state", ("load_state", "state1", True),
                                          ("load_state", "state2", False)]
        assert sorted(os.listdir(str(d))) == ["adam_m.npy", "adam_v.npy", "gradients.npy", "loss.npy", "params.npy"]
        dumps.append({f[:-4]: np.load(str(d / f)) for f in os.listdir(str(d))})
    sep = FakeRun.made[-1].sep
    assert np.array_equal(dumps[0]["loss"], np.array([0.07], np.float32)) and np.array_equal(dumps[0]["loss"], dumps[1]["loss"])
    full_params = sep.params.numpy()
    idx = np.array([int(np.flatnonzero(full_params == v)[0]) for v in dumps[0]["params"]])
    assert len(set(idx)) == 300 and (np.diff(idx) > 0).all()         # distinct elements in flat order
    for name, t in (("gradients", sep.grads), ("params", sep.params), ("adam_m", sep.adam_m), ("adam_v", sep.adam_v)):
        assert dumps[0][name].dtype == np.float32 and dumps[0][name].shape == (300,)
        assert np.array_equal(dumps[0][name], dumps[1][name])
        assert np.array_equal(dumps[0][name], t.numpy()[idx])          # the same elements of every array


def test_steps_must_be_positive_and_dump_needs_the_engine(monkeypatch, capsys):
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit) as ex:
            bench.main()
        assert ex.value.code == 2


def test_footprint_model_is_reported_only_for_the_sources_it_was_made_from(stubbed, capsys, tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "REPO", str(tmp_path))
    os.makedirs(os.path.join(str(tmp_path), "profiles"))
    model = {"source_hash": "a" * 16, "preset": "baseline_stereo", "batch": 16, "step_distinct_bytes": 7.95e9}
    with open(os.path.join(str(tmp_path), "profiles", "r2_footprint.json"), "w") as f:
        json.dump(model, f)
    monkeypatch.setattr(bench, "kernel_source_hash", lambda: "a" * 16)
    bench.run_ours(_args(no_extras=True, no_cpu_baseline=True), 0, 1, 0)
    (line,) = _lines(capsys)
    fm = line["step_footprint_model"]
    assert fm["distinct_bytes"] == 7.95e9 and abs(fm["frac_of_step"] - fm["hbm_floor_ms"] / 4.8) < 1e-12 and 0.2 < fm["frac_of_step"] < 0.3
    monkeypatch.setattr(bench, "kernel_source_hash", lambda: "b" * 16)          # other kernel sources: stale, not reported
    bench.run_ours(_args(no_extras=True, no_cpu_baseline=True), 0, 1, 0)
    (line,) = _lines(capsys)
    assert "step_footprint_model" not in line


def test_two_rank_launch_prints_one_line_and_leaves_without_exit_handlers(stubbed, capsys, tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "REPO", str(tmp_path))
    monkeypatch.setattr(bench, "kernel_source_hash", lambda: "0" * 16)
    with pytest.raises(Exited) as ex:
        bench.run_ours(_args(gpus=2), 0, 2, 0)
    assert ex.value.args == (0,)
    (line,) = _lines(capsys)
    for k in CONTRACT_KEYS + ["dp_check", "extra_configs"]:
        assert k in line, k
    assert line["n_gpus"] == 2 and line["config"]["global_batch"] == 32 and line["config"]["parallelism"] == "dp2"
    assert "cpu_baseline" not in line                            # rank 0 at N = 1 only
    assert line["extra_configs"]["m6_full_multi_instrument_b32"]["batch_per_gpu"] == 16      # 32 windows over 2 ranks
    assert "bucketed (4 buckets)" in line["config"]["allreduce"]
    main_run = FakeRun.made[0]
    assert main_run.graph is None and main_run.ar is None        # the graph (captured NCCL kernels) goes before the process group
    # the other rank: same phases, no line
    with pytest.raises(Exited):
        bench.run_ours(_args(gpus=2), 1, 2, 1)
    assert _lines(capsys) == []


def test_a_phase_that_never_returns_still_yields_the_measured_line(stubbed, capsys, monkeypatch):
    """dp_check blocks (a collective whose peer died): the guard prints the line of the finished phases and ends the process."""
    import threading
    released = threading.Event()

    def stuck(run):
        released.wait(20.0)
        raise Exited("released")
    monkeypatch.setattr(bench, "dp_check", stuck)
    real_guard = bench.LineGuard
    monkeypatch.setattr(bench, "LineGuard", lambda rank, world, seconds: real_guard(rank, world, 0.5))
    fired = []

    def fake_exit(code):                                         # called on the guard's timer thread
        fired.append(code)
        released.set()
    monkeypatch.setattr(os, "_exit", fake_exit)
    with pytest.raises(Exited):
        bench.run_ours(_args(gpus=2), 0, 2, 0)
    assert fired == [0]
    (line,) = _lines(capsys)
    assert line["aborted_in"] == "dp_check"
    for k in [k for k in CONTRACT_KEYS if k != "roofline"]:      # the per-layer roofline is filled after dp_check
        assert k in line, k
    assert abs(line["ms_per_step"] - 4.8) < 1e-9


def test_guard_is_inert_on_one_gpu_and_silent_once_disarmed(capsys, monkeypatch):
    calls = []
    monkeypatch.setattr(os, "_exit", lambda code: calls.append(code))
    g1 = bench.LineGuard(0, 1, 0.05)
    g1.update({"a": 1}, "x")
    assert g1.timer is None
    g2 = bench.LineGuard(0, 2, 0.05)
    g2.update({"a": 1}, "x")
    g2.disarm()
    time.sleep(0.2)
    assert calls == [] and capsys.readouterr().out == ""


def test_reference_arm_prints_from_rank_zero_only(monkeypatch, capsys):
    monkeypatch.setattr(bench, "cpu_step_rate", lambda cfg, budget, steps=None, warmup=1: {
        "value": 6e4, "ms_per_step": 270.0, "steps": steps, "cores": 16, "host_logical_cpus": 128, "host_physical_cores": 64,
        "sample": "stub"})
    bench.run_reference(_args(impl="reference", gpus=2), 1, 2)
    assert capsys.readouterr().out == ""
    bench.run_reference(_args(impl="reference", gpus=2), 0, 2)
    (line,) = _lines(capsys)
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["metric"] == bench.METRIC and line["unit"] == bench.UNIT
    assert line["e2e"] == {"value": line["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]


# SURVEY 8(d), per-layer live forward at M4 batch 16: GFLOP | minimal HBM MB (read input once + write live output once)
SURVEY_M4_B16 = {0: (1.887, 144.7), 1: (22.644, 239.0), 2: (33.959, 207.5), 3: (33.944, 147.7), 4: (28.262, 95.8), 5: (21.159, 58.8),
                 6: (14.759, 34.8), 7: (9.770, 20.0), 8: (6.191, 11.2), 9: (3.757, 6.1), 10: (2.159, 3.2), 11: (1.131, 1.6),
                 12: (0.388, 0.6), 13: (0.359, 0.7), 14: (0.490, 1.0), 15: (0.716, 1.6), 16: (1.087, 2.5), 17: (1.667, 4.3),
                 18: (2.526, 7.3), 19: (3.716, 12.4), 20: (5.216, 20.6), 21: (6.811, 33.2), 22: (7.937, 50.4), 23: (7.554, 69.3),
                 24: (4.531, 75.5)}


@pytest.mark.parametrize("first_layer", ["1", "0"], ids=["dedicated_first_layer", "generic_first_layer"])
def test_stack_roofline_accounting_reproduces_the_survey_table(first_layer, monkeypatch):
    """The algorithmic FLOPs and bytes behind `stack_roofline` come from the planner's own launch descriptions; for the benchmark
    configuration they must be the per-layer figures SURVEY 8(d) derived by hand from the reference's shapes - pair-merged
    launches included (the up blocks at batch 16)."""
    import Config
    import wun
    from oracle import wave_unet_oracle as O
    monkeypatch.setenv("WUN_FIRST_LAYER", first_layer)
    cfg = Config.build_config(["baseline_stereo"], experiment_id=0)["model_config"]
    t_in, _ = O.get_padding(cfg, cfg["num_frames"])
    eng = wun.Engine(wun.config_from_model_config(cfg), input_frames=t_in)
    assert any(d["launch"]["pairC"] for d in eng.launch_descriptions(16) if d["launch"]["pass"] == 0)
    peaks = {"tf_sustained": 1414.5, "hbm_gbs": 6579.6}
    sr = bench.stack_roofline(eng, 16, peaks, cfg)
    fwd = {it["layer"]: it for it in sr["items"] if it["pass"] == "fwd"}
    assert sorted(fwd) == list(range(25))
    for layer, (gf, mb) in SURVEY_M4_B16.items():
        assert abs(fwd[layer]["gflop"] - gf) < 6e-4, (layer, fwd[layer]["gflop"], gf)
        assert abs(fwd[layer]["mbytes"] - mb) < 0.06, (layer, fwd[layer]["mbytes"], mb)
    conv_fwd = sum(it["gflop"] for it in fwd.values())
    assert abs(conv_fwd + 0.027 - eng.forward_backward_flops(16) * 1e-9 / 3 - 1.887 / 3) < 0.02      # 666.1 = 3 x 222.65 - dgrad(down0)
    dg0 = [it for it in sr["items"] if it["layer"] == 0 and it["pass"] == "dgrad"][0]
    assert dg0["gflop"] == 0.0 and dg0["mbytes"] == 0.0         # no gradient w.r.t. the input waveform
    # every item is the larger of its two bounds, and the sum is what the line reports
    total = 0.0
    for it in sr["items"]:
        t_f, t_b = it["gflop"] * 1e9 / 1414.5e12, it["mbytes"] * 1e6 / 6579.6e9
        assert abs(it["us"] * 1e-6 - max(t_f, t_b)) < 1e-12 and it["bound"] == ("hbm" if t_b > t_f else "tensor")
        total += max(t_f, t_b)
    assert abs(sr["bound_ms"] - total * 1e3) < 1e-9
    adam = sr["items"][-1]
    assert adam["layer"] == "adam" and abs(adam["mbytes"] - 7 * 4 * 10263390 * 1e-6) < 1e-6      # SURVEY a15: 10 263 390 parameters
