#!/usr/bin/env python
"""bench.py - benchmarks of the B200 Wave-U-Net engine (one JSON line on stdout).

Headline metric (BASELINE.json): audio samples/sec, fwd+bwd, M4 context model.
Pinned definition (SURVEY 8(d)): OUTPUT FRAMES per second = B * T_out / step_time, a stereo frame counts once; one step =
forward + MSE loss + backward (+ NCCL gradient all-reduce when N > 1) + Adam, i.e. one `sess.run([separator_solver, ...])` of
/root/reference/Training.py:103-109, on synthetic windows (147443 in / 16389 out, stereo), batch 16 per GPU (weak scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras] [--no-graph] [--no-overlap]
                  [--dump-outputs DIR]

`--dump-outputs DIR` writes what the timed step computes from the run's seeded starting state as DIR/<name>.npy (see
dump_outputs), so that two builds can be compared output for output on identical inputs.  bench.py writes nothing into the
source tree: the per-layer table goes to the temporary directory.

The line also carries, under "extra_configs", short measurements of the other BASELINE.json configurations made in the same
run: M5 `full` (learned upsampling) batch 16, M6 `full_multi_instrument` GLOBAL batch 32 (strong scaling: 32/N windows per
GPU) and the Predict.py long-form case (3 min of 44.1 kHz stereo = 485 windows, sharded over the ranks).

Under torchrun (N > 1) the step's single collective - the all-reduce of the flat gradient buffer - runs bucketed on a
communication stream while backward still computes, and the whole step incl. NCCL is one CUDA graph.
`--impl reference` times the CPU restatement of the same step (oracle/, torch-CPU, host cores): the reference itself is
TensorFlow 1.8 and cannot be installed here (DESIGN.md).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True          # the tree may be read-only, and a benchmark run leaves it as it found it
REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "wave-u-net_b200")
for p in (REPO, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "audio samples/sec fwd+bwd, M4 context model (output frames/s)"
UNIT = "frames/s"
PRESET = "baseline_stereo"       # M4 (Config.py:71-78)
BATCH_PER_GPU = 16               # BASELINE.json configs[1]


def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(source="measured (MEASURED_PEAKS.json)", hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"],
                    tf_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]))
    return dict(source="fallback (B200_PROFILING.md)", hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0)


def host_cores():
    """(logical CPUs visible to this process, physical cores of the box or None)."""
    logical = os.cpu_count() or 1
    try:
        logical = len(os.sched_getaffinity(0))
    except Exception:
        pass
    physical = None
    try:
        import psutil
        physical = psutil.cpu_count(logical=False)
    except Exception:
        pass
    return logical, physical


def kernel_source_hash():
    """sha256 over the CUDA/C++ sources of libwun.so: ties an ncu capture under profiles/ to the build that ran."""
    h = hashlib.sha256()
    d = os.path.join(PKG, "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cpp", ".h")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        inside = [ln for (ts, ln) in self.lines if (t_begin is None or ts >= t_begin) and (t_end is None or ts <= t_end + 0.06)]
        if not inside:                       # timed region shorter than one sample: take the samples closest to it
            inside = [ln for (ts, ln) in self.lines[-2:]]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


class LineGuard(object):
    """Multi-rank runs only.  Once the timed measurement exists, nothing that follows it (per-layer table, DP check, the extra
    configurations - each holds collectives) may cost the line: if those phases do not finish within `seconds`, rank 0 prints
    the line as it stood after the last finished phase, with "aborted_in" naming the phase that did not return, and every rank
    leaves through os._exit (a rank blocked in a collective cannot unwind)."""

    def __init__(self, rank, world, seconds):
        self.rank, self.active, self.seconds = rank, world > 1, seconds
        self.lock = threading.Lock()
        self.snapshot, self.phase, self.done, self.timer = None, None, False, None

    def update(self, line, next_phase):
        """Record the line as it stands (serialised now - the caller keeps filling it) and the phase that starts next."""
        if not self.active:
            return
        try:
            snap = json.dumps(line)
        except Exception:                    # noqa: BLE001 - the guard must never be the reason a run fails
            snap = self.snapshot
        with self.lock:
            self.snapshot, self.phase = snap, next_phase
        if self.timer is None:
            self.timer = threading.Timer(self.seconds, self._fire)
            self.timer.daemon = True
            self.timer.start()

    def _fire(self):
        with self.lock:
            if self.done:
                return
            if self.rank == 0 and self.snapshot is not None:
                d = json.loads(self.snapshot)
                d["aborted_in"] = self.phase
                print(json.dumps(d), flush=True)
            sys.stderr.write("bench.py: rank %d: phase %r did not finish within %.0f s - leaving\n" % (self.rank, self.phase, self.seconds))
            sys.stderr.flush()
            os._exit(0)

    def disarm(self):
        if not self.active:
            return
        with self.lock:
            self.done = True
        if self.timer is not None:
            self.timer.cancel()


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle restatement; the only place bench.py executes oracle/ compute)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_step_rate(cfg, seconds_budget, steps=None, warmup=1):
    """Times the oracle's restatement of one Training.py:103-109 step (fwd + MSE + bwd + TF-Adam) on the
    host cores, on a bounded sample (batch 1 window per step) of the same workload."""
    import numpy as np
    import torch
    from oracle import wave_unet_oracle as O
    t_in, t_out = O.get_padding(cfg, cfg["num_frames"])
    params = O.init_params(cfg, seed=1337)
    mix, targets = O.synthetic_batch(cfg, 1, t_in, t_out, seed=1)
    m = {k: np.zeros_like(v) for k, v in params.items()}
    v = {k: np.zeros_like(p) for k, p in params.items()}

    def one(step):
        _, _, grads = O.forward_backward(cfg, params, mix, targets)
        for k in params:
            params[k], m[k], v[k] = O.adam_update(params[k], grads[k], m[k], v[k], step, 1e-4)

    # "all the host threads it can use": one window's convs do not scale past a few dozen threads (oneDNN
    # oversubscribes badly on 100+ core hosts), so pick the fastest of a few thread counts, then time with that.
    logical, physical = host_cores()
    best_t, best_n = None, 1
    for nthr in sorted(set([min(logical, c) for c in (8, 16, 32)])):     # >32 threads only loses (measured: 128 threads = 100x slower)
        torch.set_num_threads(nthr)
        one(1)
        t0 = time.perf_counter(); one(1); dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, best_n = dt, nthr
    torch.set_num_threads(best_n)
    for i in range(warmup):
        one(i + 1)
    t0 = time.perf_counter()
    n = 0
    while True:
        one(warmup + n + 1)
        n += 1
        el = time.perf_counter() - t0
        if steps is not None:
            if n >= steps:
                break
        elif el >= seconds_budget and n >= 3:
            break
    el = time.perf_counter() - t0
    return dict(value=t_out * n / el, ms_per_step=1e3 * el / n, steps=n, cores=torch.get_num_threads(),
                host_logical_cpus=logical, host_physical_cores=physical,
                sample="ONE M4 window per step (batch 1 of the batch-16 workload: 147443 in / 16389 out stereo), %d steps of "
                       "fwd+loss+bwd+Adam, normalised to output frames/s; threads = fastest of 8/16/32" % n)


def run_reference(args, rank, world):
    if rank != 0:
        return
    import Config
    cfg = Config.build_config([PRESET], experiment_id=0)["model_config"]
    r = cpu_step_rate(cfg, 0, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "M4 baseline_stereo, L=12, 147443-in/16389-out stereo; bounded sample: ONE window per step "
                                   "(the GPU arm runs 16 per GPU per step) - compare in frames/s",
                       "note": "CPU restatement (torch/oneDNN fp32) of the Training.py step, not TensorFlow 1.8"},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                             "host_logical_cpus": r["host_logical_cpus"], "host_physical_cores": r["host_physical_cores"],
                             "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
class TrainingRun(object):
    """One data-parallel training configuration: separator, device + pinned host batches, step function, graph."""

    def __init__(self, preset, local_batch, global_batch, rank, world, dev, dist, overlap=True, seed=1337):
        import numpy as np
        import torch
        import Config
        from Models.UnetAudioSeparator import UnetAudioSeparator
        from oracle import wave_unet_oracle as O     # data synthesis only (SURVEY 8(d)); not on the timed path
        self.cfg = Config.build_config([preset], experiment_id=0)["model_config"]
        self.preset, self.B, self.rank, self.world, self.dev, self.dist = preset, local_batch, rank, world, dev, dist
        self.t_in, self.t_out = O.get_padding(self.cfg, self.cfg["num_frames"])
        mix_np, targets = O.synthetic_batch(self.cfg, local_batch, self.t_in, self.t_out, seed=seed + rank)
        tg_np = np.stack([targets[s] for s in self.cfg["source_names"]])
        self.sep = UnetAudioSeparator(self.cfg)
        self.eng = self.sep.engine(input_frames=self.t_in)
        self.sep._ensure_params(self.eng, dev, create=True)      # same seed on every rank -> identical replicas (DP invariant)
        self.sep._ensure_training_state()
        self.lr = self.cfg["init_sup_sep_lr"]
        self.mix_h = torch.from_numpy(mix_np).pin_memory()
        self.tg_h = torch.from_numpy(tg_np).pin_memory()
        self.mix_d = self.mix_h.to(dev)
        self.tg_d = self.tg_h.to(dev)
        self.grad_scale = float(local_batch) / float(global_batch)
        self.global_batch = global_batch
        self.ar = None
        if world > 1 and overlap:
            from wun.parallel import BucketedAllReduce
            self.ar = BucketedAllReduce(self.eng, self.sep.grads, n_buckets=4)
        self.graph = None
        self.stream = torch.cuda.Stream(device=dev)

    def step(self):
        self.sep.loss_and_gradients(self.mix_d, self.tg_d, grad_scale=self.grad_scale)
        if self.world > 1:
            if self.ar is not None:
                self.ar.run()
            else:
                self.dist.all_reduce(self.sep.grads)
        self.sep.adam_step(self.lr)

    def prepare(self, use_graph=True):
        """Two eager steps, then capture the step (NCCL included) in a CUDA graph; falls back to eager launches."""
        import torch
        self.graph_error = None
        with torch.cuda.stream(self.stream):
            for _ in range(2):
                self.step()
            self.stream.synchronize()
            if use_graph:
                try:
                    g = torch.cuda.CUDAGraph()
                    mode = "thread_local" if self.world > 1 else "global"      # NCCL's watchdog thread polls events
                    with torch.cuda.graph(g, stream=self.stream, capture_error_mode=mode):
                        self.step()
                    self.graph = g
                except Exception as ex:                                        # noqa: BLE001
                    self.graph, self.graph_error = None, "%s: %s" % (type(ex).__name__, str(ex)[:200])
                    torch.cuda.synchronize()
        return self.graph is not None

    def run_step(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.step()

    def save_state(self):
        """Copies of what a step reads and updates in place: parameters, Adam slots, Adam's step and beta powers."""
        import torch
        s = self.sep
        state = [t.clone() for t in (s.params, s.adam_m, s.adam_v, s._adam_state)]
        torch.cuda.synchronize()             # the copies are made before the launching stream's next step
        return state

    def load_state(self, state, step=False):
        """Copies a saved state back in place (the captured step keeps its pointers); step=True: then one step."""
        import torch
        s = self.sep
        with torch.cuda.stream(self.stream):
            for t, v in zip((s.params, s.adam_m, s.adam_v, s._adam_state), state):
                t.copy_(v)
            if step:
                self.run_step()
        self.barrier()

    def barrier(self):
        import torch
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def time_steps(self, steps, warmup, prewarm_s=0.0):
        """(ms for `steps` steps as the max over ranks, perf_counter begin, end) - CUDA events on the launching stream,
        barrier + synchronize on both sides."""
        import torch
        with torch.cuda.stream(self.stream):
            if prewarm_s > 0:                # a box that has just been handed over is cold (clocks / power state): the first process on
                # it measured 2-4 % slower than the second.  A FIXED number of untimed replays (the same on every rank - the step holds a
                # collective), about prewarm_s of GPU time, then the W warm-up steps the caller asked for.
                for _ in range(int(prewarm_s / 0.006)):
                    self.run_step()
                self.stream.synchronize()
            for _ in range(warmup):
                self.run_step()
            self.stream.synchronize()
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_begin = time.perf_counter()
            e0.record(self.stream)
            for _ in range(steps):
                self.run_step()
            e1.record(self.stream)
            self.stream.synchronize()
            torch.cuda.synchronize()
            t_end = time.perf_counter()
            ms = e0.elapsed_time(e1)
        ms = self.max_over_ranks(ms)
        self.barrier()
        return ms, t_begin, t_end

    def max_over_ranks(self, x):
        import torch
        if self.world > 1:
            t = torch.tensor([float(x)], device=self.dev, dtype=torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return float(x)

    def frames_per_step(self):
        return self.global_batch * self.t_out

    def e2e(self, steps, warmup):
        """The same step through the facade with HOST buffers: every step copies its inputs from pinned host memory and
        reads its loss back.  Sequential, then with the package's prefetcher (H2D of step i+1 under the compute of step i)."""
        import torch
        out = {}
        with torch.cuda.stream(self.stream):
            def step_e2e():
                self.mix_d.copy_(self.mix_h, non_blocking=True)
                self.tg_d.copy_(self.tg_h, non_blocking=True)
                self.run_step()
                return float(self.sep._loss.item())      # device -> host read of the step's result

            for _ in range(max(1, min(3, warmup))):
                step_e2e()
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                last = step_e2e()
            torch.cuda.synchronize()
            seq_s = self.max_over_ranks(time.perf_counter() - t0)
            out.update(sequential_s=seq_s, last_loss=last, prefetch_s=None, prefetch_error=None)
            try:
                from wun.prefetch import DevicePrefetcher
                pf = DevicePrefetcher([self.mix_d, self.tg_d])

                def run_pipelined(n):
                    loss = None
                    pf.issue([self.mix_h, self.tg_h])
                    for i in range(n):
                        if i + 1 < n:
                            pf.issue([self.mix_h, self.tg_h])
                        pf.consume()
                        self.run_step()
                        loss = float(self.sep._loss.item())
                    return loss

                run_pipelined(max(2, min(3, warmup)))
                self.barrier()
                t0 = time.perf_counter()
                pipe_loss = run_pipelined(steps)
                torch.cuda.synchronize()
                pipe_s = self.max_over_ranks(time.perf_counter() - t0)
                if not (pipe_loss == pipe_loss and 0.0 < pipe_loss < 10.0):      # finite, plausible MSE
                    raise RuntimeError("implausible loss %r from the pipelined loop" % (pipe_loss,))
                out["prefetch_s"] = pipe_s
                if pipe_s < seq_s:
                    out["last_loss"] = pipe_loss
            except Exception as ex:                                               # noqa: BLE001 - keep the bench line alive
                out["prefetch_error"] = "%s: %s" % (type(ex).__name__, ex)
        out["bytes_h2d"] = int(self.mix_h.numel() * 4 + self.tg_h.numel() * 4)
        return out


DUMP_SAMPLE = 3000000          # elements kept of each parameter-sized array: 4 x 12 MB, within the dump's 64 MB


def dump_outputs(run, out_dir):
    """What the step run last handed its caller, as float32 DIR/<name>.npy: the loss, and the gradients and the parameters and
    Adam slots after its update.  Of these four parameter-sized arrays (10.3 M elements for M4) the same fixed sample is kept
    (sorted flat indices, seed 0) - all of them when a model has at most DUMP_SAMPLE parameters."""
    import numpy as np
    import torch
    sep = run.sep
    torch.cuda.synchronize()
    n = sep.params.numel()
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    idx = torch.from_numpy(idx).to(sep.params.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), sep._loss.detach().cpu().numpy().astype(np.float32))
    for name, t in (("gradients", sep.grads), ("params", sep.params), ("adam_m", sep.adam_m), ("adam_v", sep.adam_v)):
        np.save(os.path.join(out_dir, name + ".npy"), t[idx].cpu().numpy().astype(np.float32))


def layer_table(run, iters=6):
    """Every conv layer x pass (fwd, dgrad, wgrad) timed ALONE with CUDA events on the launching stream, on the tensors the
    last training step left in the workspace (Engine.run_layer_pass).  Returns (rows, families)."""
    import torch
    L = run.cfg["num_layers"]
    names = ["down%d" % i for i in range(L)] + ["bottleneck"] + ["up%d" % i for i in range(L)]
    scratch = torch.zeros_like(run.sep.grads)
    rows = []
    with torch.cuda.stream(run.stream):
        for layer in range(2 * L + 1):
            for pass_, pname in ((0, "fwd"), (1, "dgrad"), (2, "wgrad")):
                if pass_ == 1 and layer == 0:
                    continue                                  # no gradient w.r.t. the input waveform
                fl = run.eng.run_layer_pass(layer, pass_, 2, run.sep.params, run.mix_d, scratch)      # warm-up
                run.stream.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(run.stream)
                if layer == 0 and pass_ == 0:
                    # the library repeats only a tensor-core conv `iters` times inside one call (pack once, launch often); the first
                    # layer has its own kernels, launched once per call - repeat the call instead (round-2 lines divided one launch by 6)
                    for _ in range(iters):
                        run.eng.run_layer_pass(layer, pass_, 1, run.sep.params, run.mix_d, scratch)
                else:
                    run.eng.run_layer_pass(layer, pass_, iters, run.sep.params, run.mix_d, scratch)
                e1.record(run.stream)
                run.stream.synchronize()
                us = e0.elapsed_time(e1) * 1e3 / iters
                rows.append({"layer": names[layer], "pass": pname, "us": us, "gflop": fl * 1e-9,
                             "tflops": (fl / (us * 1e-6) * 1e-12) if us > 0 else 0.0})
    fam = {}
    for r in rows:
        key = "first_layer" if r["layer"] == "down0" else {"fwd": "conv_fwd", "dgrad": "conv_dgrad", "wgrad": "wgrad"}[r["pass"]]
        f = fam.setdefault(key, {"us": 0.0, "gflop": 0.0, "launch_groups": 0})
        f["us"] += r["us"]; f["gflop"] += r["gflop"]; f["launch_groups"] += 1
    for f in fam.values():
        f["tflops"] = f["gflop"] * 1e9 / (f["us"] * 1e-6) * 1e-12 if f["us"] > 0 else 0.0
    return rows, fam


def account_launch(d):
    """(FLOPs, input elements, output elements) PER BATCH ITEM of one exported forward plane-convolution launch
    (Engine.launch_descriptions): 2 FLOP per MAC over the rows the classes write; input = the rows of every distinct plane view the
    terms actually read, once; output = the rows written, once - SURVEY 8(d)'s "minimal HBM bytes = read input once + write live
    output once" (tests/test_bench_contract.py checks the M4 table against SURVEY's per-layer figures)."""
    L, planes, pairC = d["launch"], d["planes"], d["launch"]["pairC"]
    flops, out_el, span = 0, 0, {}
    for q in d["cls"]:
        if q["m_hi"] <= q["m_lo"]:
            continue
        out_el += (((q["hi0"] - q["lo0"]) + (q["hi1"] - q["lo1"])) * pairC) if pairC else (q["m_hi"] - q["m_lo"]) * L["N"]
        for t in d["terms"][q["term_begin"]:q["term_end"]]:
            P = planes[t["plane"]]
            if pairC:
                rows = (q["hi0"] - q["lo0"] if t["woff"] >= 0 else 0) + (q["hi1"] - q["lo1"] if t["woff2"] >= 0 else 0)
                flops += 2 * P["C"] * pairC * rows
            else:
                flops += 2 * P["C"] * L["N"] * (q["m_hi"] - q["m_lo"])
            a, b = max(P["r_lo"], q["m_lo"] + t["d"]), min(P["r_hi"], q["m_hi"] + t["d"])
            if b > a:
                b += 1 if P["kind"] == 1 else 0                  # an interpolated row reads its successor too
                key = (P["base"], P["rstride"])                  # the copied and the interpolated plane of an up block share their tensor
                lo, hi, _ = span.get(key, (a, b, 0))
                span[key] = (min(lo, a), max(hi, b), P["C"])
    return flops, sum((hi - lo) * C for lo, hi, C in span.values()), out_el


def stack_roofline(eng, batch, peaks, cfg):
    """SURVEY 8(d): "the stack bound is the sum over layers of max(FLOPs / peak, bytes / BW)" - the per-layer conv arithmetic
    roofline of one training step (forward, dgrad, wgrad of every conv layer + the Adam pass), from the planner's own launch
    descriptions (host-only dry run).  Bytes per layer and pass: forward in + out, dgrad out + 2 in (gradient in, saved activation
    for the slope, gradient out), wgrad in + out; Adam reads p, g, m, v and writes p, m, v."""
    import ctypes
    import wun
    fwd = {d["launch"]["layer"]: account_launch(d) for d in eng.launch_descriptions(batch) if d["launch"]["pass"] == 0}
    n_layers = 2 * cfg["num_layers"] + 1
    if 0 not in fwd:                                             # the first layer has its own kernels: no plane-convolution launch
        rows_out = 0
        for name in ("dec0", "odd0"):
            off, rows, ch = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int32()
            wun.check(wun.lib.wun_debug_tensor(eng._h, name.encode(), int(batch), 1, ctypes.byref(off), ctypes.byref(rows), ctypes.byref(ch)))
            rows_out += rows.value * ch.value
        c_in = 1 if cfg["mono_downmix"] else 2
        f0 = 2 * rows_out * cfg["filter_size"] * c_in
        fwd[0] = (f0, eng.T_in * c_in, rows_out)
    p_tensor, bw = peaks["tf_sustained"] * 1e12, peaks["hbm_gbs"] * 1e9
    items, t_sum, t_sum3, f_sum = [], 0.0, 0.0, 0.0
    for layer in range(n_layers):
        f, i_el, o_el = (x * batch for x in fwd[layer])
        for pname, fl, by in (("fwd", f, 4 * (i_el + o_el)), ("dgrad", f if layer > 0 else 0, 4 * (o_el + 2 * i_el) if layer > 0 else 0),
                              ("wgrad", f, 4 * (i_el + o_el))):
            t_f, t_b = fl / p_tensor, by / bw
            items.append({"layer": layer, "pass": pname, "gflop": fl * 1e-9, "mbytes": by * 1e-6, "bound": "hbm" if t_b > t_f else "tensor",
                          "us": max(t_f, t_b) * 1e6})
            t_sum += max(t_f, t_b)
            t_sum3 += max(3.0 * t_f, t_b)                        # the fp32-accurate scheme issues 3 bf16 MMAs per product
            f_sum += fl
    adam_bytes = 7 * 4 * eng.param_numel
    items.append({"layer": "adam", "pass": "update", "gflop": 0.0, "mbytes": adam_bytes * 1e-6, "bound": "hbm", "us": adam_bytes / bw * 1e6})
    t_sum += adam_bytes / bw
    t_sum3 += adam_bytes / bw
    return {"bound_ms": t_sum * 1e3, "bound_ms_3mma": t_sum3 * 1e3, "gflop": f_sum * 1e-9,
            "hbm_bound_passes": sum(1 for it in items if it["bound"] == "hbm"), "passes": len(items), "items": items}


def dp_check(run):
    """Hardware data-parallel correctness (SURVEY section 4 item 6), run on the benchmark's own replicas:
      (a) the replicas are still bit-identical after all the Adam steps of this run;
      (b) the all-reduced gradient of the sharded batch == the gradient ONE GPU computes for the concatenated batch."""
    import torch
    dist, world, dev = run.dist, run.world, run.dev
    sep = run.sep
    torch.cuda.synchronize()
    h = torch.stack([sep.params.view(torch.int32).to(torch.int64).sum(),
                     sep.adam_v.view(torch.int32).to(torch.int64).sum()])
    hs = [torch.empty_like(h) for _ in range(world)]
    dist.all_gather(hs, h)
    identical = all(bool(torch.equal(hs[0], x)) for x in hs)
    nb = min(2, run.B)                                    # windows per rank used for (b)
    mix_l = run.mix_d[:nb].contiguous()
    tg_l = run.tg_d[:, :nb].contiguous()
    sep.loss_and_gradients(mix_l, tg_l, grad_scale=1.0 / world)
    dist.all_reduce(sep.grads)
    g_dp = sep.grads.clone()
    mixes = [torch.empty_like(mix_l) for _ in range(world)]
    tgs = [torch.empty_like(tg_l) for _ in range(world)]
    dist.all_gather(mixes, mix_l)
    dist.all_gather(tgs, tg_l)
    rel = rel_sum = None
    if run.rank == 0:
        # (b1) communication alone: the same shards, each at the per-rank batch size, summed on ONE GPU - identical kernels, so only
        #      the summation order of the all-reduce differs (fp32 noise)
        g_sum = torch.zeros_like(g_dp)
        for m_r, t_r in zip(mixes, tgs):
            sep.loss_and_gradients(m_r.contiguous(), t_r.contiguous(), grad_scale=1.0 / world)
            g_sum += sep.grads
        rel_sum = float(((g_dp - g_sum).double().norm() / g_sum.double().norm()).item())
        # (b2) the concatenated batch in one call: other tilings (the planner's choices depend on the batch), so a pre-activation
        #      within rounding noise of zero can take the other LeakyReLU slope - the bar is the parity tests' 1e-3 (tests/test_gpu_parity.py)
        sep.loss_and_gradients(torch.cat(mixes, 0).contiguous(), torch.cat(tgs, 1).contiguous(), grad_scale=1.0)
        g_one = sep.grads
        rel = float(((g_dp - g_one).double().norm() / g_one.double().norm()).item())
    dist.barrier()
    return {"replicas_identical_after_adam": identical, "allreduced_grad_vs_sum_of_shard_grads_rel_l2": rel_sum,
            "allreduced_grad_vs_single_gpu_rel_l2": rel, "windows_per_rank": nb,
            "ok": bool(identical and (rel is None or (rel < 1e-3 and rel_sum < 1e-5)))}


def predict_bench(rank, world, dev, dist, reps=2):
    """BASELINE.json config 5: Predict.py long-form inference - 3 min of 44.1 kHz stereo through Evaluate.predict_track
    (device-side window gather / batched forward / scatter, windows sharded over the ranks), host array in, host arrays out."""
    import numpy as np
    import torch
    import Config
    import Evaluate
    from Models.UnetAudioSeparator import UnetAudioSeparator
    cfg = Config.build_config(["full_44KHz"], experiment_id=0)["model_config"]
    n_frames = 180 * 44100
    rng = np.random.default_rng(1337)
    audio = (rng.uniform(-1.0, 1.0, size=(n_frames, 2)) * 0.5).astype(np.float32)
    sep = UnetAudioSeparator(cfg)
    in_shape, out_shape = sep.get_padding(np.array([1, cfg["num_frames"], 0]))
    eng = sep.engine(input_frames=int(in_shape[1]))
    sep._ensure_params(eng, dev, create=True)
    n_windows = len(Evaluate.window_starts(n_frames, int(out_shape[1])))
    best = None
    for i in range(reps + 1):                              # first pass = warm-up (workspace allocation)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        preds = Evaluate.predict_track(cfg, sep, audio, batch_windows=16, device=dev)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        if i > 0:
            best = dt if best is None else min(best, dt)
    assert preds[cfg["source_names"][0]].shape == (n_frames, 2)
    return {"workload": "Predict: 3 min 44.1 kHz stereo, preset full_44KHz (M5-HighSR), %d windows of 147443 frames, 16 per "
                        "batch, sharded over %d GPU(s); host array in, host arrays out" % (n_windows, world),
            "seconds": best, "audio_seconds_per_s": 180.0 / best, "frames_per_s": n_frames / best, "windows": n_windows,
            "n_gpus": world}


def run_ours(args, rank, world, local_rank):
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()                       # samples are time-stamped; only those inside the timed region are reported
    run = TrainingRun(PRESET, BATCH_PER_GPU, BATCH_PER_GPU * world, rank, world, dev, dist, overlap=not args.no_overlap)
    start = run.save_state() if args.dump_outputs else None
    graphed = run.prepare(use_graph=not args.no_graph)
    ms_total, t_begin, t_end = run.time_steps(args.steps, args.warmup, prewarm_s=0.0 if args.no_prewarm else 1.5)
    clk = clocks.stop(t_begin, t_end) if rank == 0 else None
    if args.dump_outputs:
        # The state after hundreds of steps is not reproducible: the weight-gradient reductions add in a varying order and Adam
        # amplifies those last-bit differences (two default runs on a B200, ~300 steps each: final gradients 0.8 apart in rel. L2).
        # So the timed step runs once more, after the timing, from the seeded starting state, and that step's results are written.
        timed = run.save_state()
        run.load_state(start, step=True)
        if rank == 0:
            dump_outputs(run, args.dump_outputs)
        run.load_state(timed)                # the phases below continue from where the timed steps left off
    e_steps = max(3, min(args.steps, 10))
    e2e = run.e2e(e_steps, args.warmup)

    ms_step = ms_total / args.steps
    frames = run.frames_per_step()
    value = frames / (ms_step * 1e-3)
    e2e_s = min(e2e["sequential_s"], e2e["prefetch_s"]) if e2e["prefetch_s"] else e2e["sequential_s"]
    e2e_value = frames / (e2e_s / e_steps)
    peaks = load_peaks()
    flops = run.eng.forward_backward_flops(run.B)
    step_tf = flops / (ms_step * 1e-3) * 1e-12

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "input_frames_per_s": value * run.t_in / run.t_out,      # SURVEY 8(d): the same rate counted in input frames (x 8.997 for M4)
        "config": {"workload": "M4 baseline_stereo L=12, 147443-in/16389-out stereo, batch %d per GPU, "
                               "fwd+loss+bwd+Adam%s" % (run.B, "+NCCL all-reduce" if world > 1 else ""),
                   "global_batch": run.B * world, "parallelism": "dp%d" % world,
                   "l2_policy": "per-step working set (~1.2 GB activations + gradients) exceeds the 126 MB L2",
                   "cuda_graph": graphed, "cuda_graph_error": run.graph_error,
                   "untimed_prewarm_steps": 0 if args.no_prewarm else int(1.5 / 0.006),
                   "allreduce": (("bucketed (%d buckets) on a comm stream, overlapped with backward" % len(run.ar.views))
                                 if run.ar is not None else "one flat all-reduce after backward") if world > 1 else None,
                   "arithmetic": "fp32 in/out; tensor-core layers split every fp32 operand into bf16 hi+lo and issue "
                                 "3 bf16 MMAs per product (fp32 accumulate): 5e-6 rel. error vs the 1e-4 parity bar"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e["bytes_h2d"], "d2h_bytes_per_step": 4,
                "steps": e_steps, "last_loss": e2e["last_loss"],
                "sequential_value": frames / (e2e["sequential_s"] / e_steps),
                "prefetch_value": (frames / (e2e["prefetch_s"] / e_steps)) if e2e["prefetch_s"] else None,
                "mode": "prefetch (wun.prefetch.DevicePrefetcher: H2D of step i+1 overlaps step i)"
                        if (e2e["prefetch_s"] and e2e["prefetch_s"] <= e2e["sequential_s"]) else "sequential",
                "prefetch_error": e2e["prefetch_error"]},
        "gpu_launches": int((run.eng.launches(True) + 2) * args.steps),
        "clocks": clk,
        "step_roofline": {"bound": "tensor", "achieved": step_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                          "frac": step_tf / peaks["tf_sustained"],
                          "scope": "whole step: %.1f algorithmic GFLOP (fwd+bwd, live positions) / step time; peak = bf16 "
                                   "sustained, %s; the fp32-accurate 3-MMA scheme caps frac at 1/3" % (flops * 1e-9, peaks["source"])},
    }
    guard = LineGuard(rank, world, 240.0)
    guard.update(line, "per-layer table")
    # ---- per-layer / per-family table: every conv layer and pass timed alone (rank 0; the others wait) -----------------
    rows, fam = None, None
    if rank == 0:
        rows, fam = layer_table(run)
    if world > 1:
        dist.barrier()
    guard.update(line, "dp_check")
    dpc = dp_check(run) if world > 1 else None
    if dpc is not None:
        line["dp_check"] = dpc
    if rank == 0:
        try:                                  # host-only accounting; never worth losing the line for
            import wun
            acct = wun.Engine(wun.config_from_model_config(run.cfg), input_frames=run.t_in)      # its own handle: a dry run only
            sr = stack_roofline(acct, run.B, peaks, run.cfg)
            del acct
            line["stack_roofline"] = {
                "bound_ms": sr["bound_ms"], "frac": sr["bound_ms"] / ms_step, "bound_ms_3mma": sr["bound_ms_3mma"],
                "frac_3mma": sr["bound_ms_3mma"] / ms_step, "gflop": sr["gflop"],
                "hbm_bound_passes": sr["hbm_bound_passes"], "passes": sr["passes"],
                "definition": "SURVEY 8(d): sum over the conv layers x (fwd, dgrad, wgrad) + Adam of max(algorithmic FLOPs / bf16 "
                              "sustained peak, algorithmic bytes / HBM bandwidth), %s; frac = that bound / measured step time; "
                              "_3mma: tensor terms x 3 (the fp32-accurate scheme issues 3 bf16 MMAs per product)" % peaks["source"]}
        except Exception as ex:               # noqa: BLE001
            line["stack_roofline"] = {"error": "%s: %s" % (type(ex).__name__, str(ex)[:200])}
    if rank == 0:
        try:                                  # the launch-footprint model of tools/footprint_model.py, if it was made for these sources
            fj = json.load(open(os.path.join(REPO, "profiles", "r2_footprint.json")))
            if fj.get("source_hash") == kernel_source_hash() and fj.get("batch") == run.B and fj.get("preset") == PRESET:
                floor_ms = fj["step_distinct_bytes"] / (peaks["hbm_gbs"] * 1e9) * 1e3
                line["step_footprint_model"] = {
                    "distinct_bytes": fj["step_distinct_bytes"], "hbm_floor_ms": floor_ms, "frac_of_step": floor_ms / ms_step,
                    "note": "sum over the launches of one step of the distinct bytes each launch touches (decoded from the engine's real "
                            "launch parameters on the host, tools/footprint_model.py) / measured HBM bandwidth: the HBM floor of the step AS "
                            "IMPLEMENTED (split arrays and weight packs included); a model, not an ncu measurement"}
        except Exception:                     # noqa: BLE001
            pass
    if rank == 0 and fam:
        dom = max((k for k in fam if k != "first_layer"), key=lambda k: fam[k]["us"])
        top = max(rows, key=lambda r: r["us"])
        traffic, traffic_note = None, "no ncu capture for this build under profiles/"
        tpath = os.path.join(REPO, "profiles", "r2_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            if tj.get("source_hash") == kernel_source_hash():
                traffic, traffic_note = tj.get("dram_bytes_per_launch", {}).get(dom), tj.get("note")
            else:
                traffic_note = "profiles/r2_traffic.json was captured on other kernel sources (%s) - stale, not reported" % tj.get("source_hash")
        line["roofline"] = {
            "bound": "tensor", "achieved": fam[dom]["tflops"], "peak": peaks["tf_burst"], "unit": "TFLOP/s",
            "frac": fam[dom]["tflops"] / peaks["tf_burst"], "traffic": traffic, "traffic_note": traffic_note,
            "kernel": "time-dominant kernel family '%s': %d layer launches, %.1f us and %.1f algorithmic GFLOP per step "
                      "(live positions, 2 FLOP/MAC, the 3 bf16 MMAs per product count once), each layer timed alone with CUDA "
                      "events" % (dom, fam[dom]["launch_groups"], fam[dom]["us"], fam[dom]["gflop"]),
            "peak_source": "bf16 dense burst, %s; the fp32-accurate 3-MMA scheme caps frac at 1/3" % peaks["source"]}
        line["families"] = {k: {"us": round(v["us"], 1), "gflop": round(v["gflop"], 2), "tflops": round(v["tflops"], 1),
                                "frac_of_burst": round(v["tflops"] / peaks["tf_burst"], 4)} for k, v in fam.items()}
        line["top_launch"] = {"layer": top["layer"], "pass": top["pass"], "us": round(top["us"], 1),
                              "gflop": round(top["gflop"], 2), "frac_of_burst": round(top["tflops"] / peaks["tf_burst"], 4)}
        try:
            path = os.path.join(tempfile.gettempdir(), "wun_bench_layer_table_n%d.json" % world)
            with open(path, "w") as f:
                json.dump({"source_hash": kernel_source_hash(), "ms_per_step": ms_step, "rows": rows, "families": fam}, f, indent=1)
            sys.stderr.write("bench.py: per-layer table written to %s\n" % path)
        except Exception:
            pass

    # ---- the other BASELINE.json configurations, briefly, in the same run ----------------------------------------------
    if not args.no_extras:
        guard.update(line, "extra_configs: M6 full_multi_instrument, global batch 32")
        extras = {}
        del run.graph
        run.graph = None
        x_steps, x_warm = 10, 3

        def train_extra(preset, local_b, global_b, scaling):
            r = TrainingRun(preset, local_b, global_b, rank, world, dev, dist, overlap=not args.no_overlap, seed=4242)
            g = r.prepare(use_graph=not args.no_graph)
            ms, _, _ = r.time_steps(x_steps, x_warm)
            fl = r.eng.forward_backward_flops(local_b) * world
            out = {"preset": preset, "global_batch": global_b, "batch_per_gpu": local_b, "n_gpus": world, "scaling": scaling,
                   "ms_per_step": ms / x_steps, "frames_per_s": r.frames_per_step() / (ms / x_steps * 1e-3),
                   "step_tflops_per_gpu": fl / world / (ms / x_steps * 1e-3) * 1e-12, "cuda_graph": g, "steps": x_steps}
            del r
            torch.cuda.empty_cache()
            return out

        try:
            line["extra_configs"] = extras
            if 32 % world == 0:
                extras["m6_full_multi_instrument_b32"] = train_extra("full_multi_instrument", 32 // world, 32, "strong")
            guard.update(line, "extra_configs: M5 full, batch 16 per GPU")
            extras["m5_full_learned_b16"] = train_extra("full", 16, 16 * world, "weak")
            guard.update(line, "extra_configs: Predict 3 min 44.1 kHz")
            extras["predict_3min_44k"] = predict_bench(rank, world, dev, dist)
        except Exception as ex:                                                    # noqa: BLE001
            extras["error"] = "%s: %s" % (type(ex).__name__, str(ex)[:300])
        line["extra_configs"] = extras

    guard.disarm()
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            cfg = run.cfg
            r = cpu_step_rate(cfg, 12.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                    "host_logical_cpus": r["host_logical_cpus"],
                                    "host_physical_cores": r["host_physical_cores"], "sample": r["sample"]}
        print(json.dumps(line), flush=True)
    # Teardown.  The step graph holds captured NCCL kernels: it goes first, then the process group.  A watchdog ends the process if
    # the teardown itself gets stuck (seen once at N=2: both workers idle after rank 0 had printed its line, until the caller's
    # timeout) - the measurement is complete and printed at this point.
    watchdog = threading.Timer(45.0, lambda: os._exit(0))
    watchdog.daemon = True
    watchdog.start()
    try:
        run.graph = None
        run.ar = None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
    finally:
        watchdog.cancel()
    if world > 1:
        # multi-rank: leave without the interpreter's exit handlers (NCCL / CUDA-graph destructors at shutdown are the other place
        # a finished run could sit until the launcher's timeout); everything is printed and flushed, the process group is gone.
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: one flat all-reduce after backward")
    ap.add_argument("--no-extras", action="store_true", help="skip the M5 / M6 / Predict measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prewarm", action="store_true", help="skip the untimed pre-warm replays (profiler runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timing, run the timed step once more from the seeded starting state; write its results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the engine's outputs: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
