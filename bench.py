#!/usr/bin/env python
"""bench.py -- body2hand frames/sec on B200 (contract: see the task statement / DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Headline workload (N GPUs): BASELINE.json config 3/4 -- the training step (forward + mask_output +
maskedPoseL1 + backward + Adam) on batch 256 x 64 frames per GPU, C=30, synthetic How2Sign-shaped
windows; weak scaling (per-GPU batch fixed) with one gradient all-reduce per step.  The same JSON line
also carries config 2 (forward, batch 512 x 64, bf16 tensor-core path) under "fwd" and the K0
preprocessing throughput under "preprocess" (N=1 only).  One JSON line on stdout (rank 0)."""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C, T, B_TRAIN, B_FWD, LR = 30, 64, 256, 512, 2e-4
S_MAC = 24 * C + 2 * C * C + 42 * C                          # MAC per tap per frame (SURVEY.md §8)
FWD_FLOP_PER_WINDOW = 2 * (5 * T - 6) * S_MAC                # 2 373 840 at T=64, C=30
TRAIN_FLOP_PER_WINDOW = 2 * (5 * T - 6) * (3 * S_MAC - 24 * C)   # 6 669 360
PRE_BYTES_PER_FRAME = 804 + 648                              # K0 figure of record (SURVEY.md §8d)
N_SLOTS = 40                                                 # resident batches rotated so the working set > L2


def dp_parity_check(b2h, synthetic, DataParallelTrainer, TrainStepRunner, dev, rank, world, prec, exchange, multicast):
    """SURVEY 8e parity, run inside the N>1 bench because the GPU test box has one GPU: W ranks x 16 windows ==
    one rank on the concatenated 16*W windows (loss per step, post-step weights), replicas bit-identical."""
    import torch
    import torch.distributed as dist
    from hand_pose_sl_b200 import parallel
    Bp, Tp, steps = 16, 64, 4
    batch = synthetic.model_batch(Bp * world, Tp, seed=77, ragged=True)
    torch.manual_seed(0)
    m = b2h.ConvModel(C, "ReLU", False, precision=prec).to(dev)
    o = b2h.FusedAdam(m.parameters(), lr=LR)
    tr = DataParallelTrainer(m, o, Bp, Tp, "L1", exchange=exchange, multicast=multicast)
    tr.load(parallel.shard_batch(batch, rank, world), non_blocking=False)
    losses = [float(parallel.combine_losses(tr.step(0), "L1")) for _ in range(steps)]
    identical = bool(tr.replicas_identical())
    tr.finish()
    flat = m.flat_parameters().clone()
    out = {"small_run": f"{world} ranks x {Bp} windows x {Tp} frames, {steps} steps, ragged lengths",
           "replicas_bit_identical": identical}
    if rank == 0:
        torch.manual_seed(0)
        ref = b2h.ConvModel(C, "ReLU", False, precision=prec).to(dev)
        ro = b2h.FusedAdam(ref.parameters(), lr=LR)
        rr = TrainStepRunner(ref, ro, Bp * world, Tp, "L1")
        rr.load(batch, non_blocking=False)
        rl = [float(rr.step(0)) for _ in range(steps)]
        rr.finish()
        rf = ref.flat_parameters()
        out["loss_rel_err_vs_1rank"] = max(abs(a - b) / abs(b) for a, b in zip(losses, rl))
        out["weights_max_abs_diff_vs_1rank"] = float((flat - rf).abs().max())
        out["weights_frac_within_1e-4"] = float(((flat - rf).abs() <= 1e-4 * rf.abs().max()).float().mean())
        out["weights_bound_2_lr_steps"] = 2 * LR * steps
    dist.barrier()
    return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tflops_burst": d["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_reference_arm(steps, warmup, budget_s=None):
    """The reference's CPU path for the headline config: its ConvModel + mask_output + maskedPoseL1 + Adam
    (restated in oracle/b2h_oracle.py from traintest.py:87-123; the reference is pure Python/PyTorch, nothing
    to compile -> kind 'port'), all host threads, same seeded batch.  With `budget_s`, stops early once the
    timed steps have taken that long."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import b2h_oracle as oracle
    from hand_pose_sl_b200 import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    batch = synthetic.model_batch(B_TRAIN, T, seed=1234)
    st = oracle.TrainState(oracle.init_params(C, False, seed=0), lr=LR)
    for _ in range(max(1, warmup)):
        oracle.train_step(st, batch["input_kp"], batch["target_kp"], batch["n_frames"])
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        oracle.train_step(st, batch["input_kp"], batch["target_kp"], batch["n_frames"])
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    # SURVEY 8d: also the "loops vectorised" variant (closed-form masked L1, one multiply for mask_output), so the
    # reader can see how much of the CPU number is the reference's per-sample Python loops
    vec_ms = None
    try:
        lens = torch.as_tensor(batch["n_frames"], dtype=torch.int64)
        keep = (torch.arange(T)[None, :] < lens[:, None]).float()[:, :, None, None]
        n_vec = max(3, min(done, 40))
        t1 = time.perf_counter()
        for _ in range(n_vec):
            pred = oracle.conv_model_forward(st.params, batch["input_kp"], st.pos_emb) * keep
            loss = oracle.masked_pose_l1_closed_form(pred, batch["target_kp"], batch["n_frames"])
            st.opt.zero_grad()
            loss.backward()
            st.opt.step()
        vec_ms = (time.perf_counter() - t1) / n_vec * 1e3
    except Exception:
        vec_ms = None
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"value": done * B_TRAIN * T / dt, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{done} train steps of batch {B_TRAIN}x{T} (C={C}, fp32, reference per-sample loss loops) in {dt:.2f} s",
            "threads": torch.get_num_threads(), "cpu": model, "ms_per_step": dt / done * 1e3,
            "ms_per_step_loops_vectorised": vec_ms,
            "value_loops_vectorised": (B_TRAIN * T / (vec_ms * 1e-3)) if vec_ms else None}, done, dt


def dump_outputs(out_dir, loss, model):
    """What the last timed train step hands its caller, as float32 .npy files: the step's loss (`loss.npy`) and the
    updated parameters (`<state-dict key>.npy`).  The inputs are seeded, so two builds run with the same arguments can
    be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.reshape(1), **model.state_dict()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_reference(args, rank):
    if rank != 0:
        return
    base, done, dt = cpu_reference_arm(args.steps, args.warmup)
    line = {"impl": "reference", "metric": "body2hand_train_frames_per_sec", "value": base["value"], "unit": "frames/s",
            "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": dt / done * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"train step (fwd+mask+L1+bwd+Adam), batch {B_TRAIN}x{T} frames, C={C} (BASELINE config 3)",
                       "global_batch": B_TRAIN, "frames_per_window": T, "conv_channels": C},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    global B_TRAIN
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "bf16", "fp32-ffma"])
    ap.add_argument("--skip-extras", action="store_true", help="only the headline train-step number")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"], help="multi-GPU gradient exchange")
    ap.add_argument("--no-multicast", action="store_true", help="p2p exchange: unicast stores even when an NVLS mapping exists")
    ap.add_argument("--strong", action="store_true", help="strong scaling (SURVEY 8d config 4): the GLOBAL batch stays 256 windows, "
                                                         "each of the N ranks trains 256/N; the default (and the driver's contract) is weak")
    ap.add_argument("--no-numa-bind", action="store_true", help="leave the rank's threads / pinned buffers where the OS puts them")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's loss and the updated "
                                                          "parameters to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 train step (--impl b200)")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.strong:
        if 256 % world:
            raise SystemExit("--strong needs a rank count that divides 256")
        B_TRAIN = 256 // world

    import torch
    import torch.distributed as dist
    import hand_pose_sl_b200 as b2h
    from hand_pose_sl_b200 import _lib, synthetic
    from hand_pose_sl_b200.parallel import DataParallelTrainer
    from hand_pose_sl_b200.runner import ForwardRunner, TrainStepRunner

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: hand_pose_sl_b200 has no CPU path (use --impl reference for the CPU arm)")
    # libraries (NCCL's version banner, ...) write to stdout; keep fd 1 clean for the ONE JSON line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    # before the first pinned allocation: the rank's threads and staging buffers go to its GPU's NUMA node
    from hand_pose_sl_b200.hostbind import bind_host_to_gpu
    # (N = 1 is left alone: the same process times the CPU baseline afterwards on ALL host cores)
    if args.no_numa_bind or world == 1:
        host_numa = {"bound": False, "why": "--no-numa-bind" if args.no_numa_bind else "single process"}
    else:
        host_numa = bind_host_to_gpu(local_rank)
    if world > 1:
        sys.stderr.write(f"[bench] rank {rank}: host placement {host_numa}\n")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it (its lines go to stderr: fd 1 is redirected below until the JSON line)
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    train_prec = "bf16" if args.precision == "auto" else args.precision
    fwd_prec = "bf16" if args.precision == "auto" else args.precision

    # ---------------- headline: training step, batch 256 x 64 per GPU ----------------
    torch.manual_seed(0)
    model = b2h.ConvModel(C, "ReLU", False, precision=train_prec).to(dev)
    opt = b2h.FusedAdam(model.parameters(), lr=LR)
    # bf16 mode ships input_kp as bf16 (the kernel rounds it to bf16 anyway: bit-identical result, shorter H2D copy)
    x_dt = torch.bfloat16 if train_prec == "bf16" else torch.float32
    if world > 1:
        runner = DataParallelTrainer(model, opt, B_TRAIN, T, "L1", n_slots=N_SLOTS, exchange=args.exchange, x_dtype=x_dt,
                                     multicast=not args.no_multicast)
    else:
        runner = TrainStepRunner(model, opt, B_TRAIN, T, "L1", n_slots=N_SLOTS, x_dtype=x_dt)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                       # long before the timed region: nvidia-smi needs ~0.2 s to start
    staged = []
    for s in range(N_SLOTS):
        b = synthetic.model_batch(B_TRAIN, T, seed=1234 + 1000 * rank + s)
        staged.append(runner.host_stage(b))                   # ONE pinned buffer per batch (x | target | lengths)
        runner.load_staged(staged[-1], slot=s, non_blocking=False)
    chunk = min(N_SLOTS, args.steps)
    graphed = True
    try:
        runner.capture(chunk)
    except Exception as e:                                    # e.g. capture refused: direct launches instead
        graphed = False
        sys.stderr.write(f"[bench] CUDA graph capture unavailable ({type(e).__name__}: {e}); direct launches\n")
        torch.cuda.synchronize()

    def run_steps(n):
        done = 0
        if graphed:
            while done + chunk <= n:
                runner.replay()
                done += chunk
        while done < n:
            runner.step(done % N_SLOTS)
            done += 1

    # warm-up: the SAME graph that is timed, at least W steps and at least one full replay
    run_steps(max(args.warmup, chunk))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    run_steps(args.steps)                                     # untimed, not synchronised: the ranks meet inside these steps
    ev0.record()                                              # ... so every rank's clock starts in lock-step with its peers
    run_steps(args.steps)
    ev1.record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:                       # before the steps below move the weights on
        dump_outputs(args.dump_outputs, runner.loss[(args.steps - 1) % N_SLOTS], model)
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    timed_steps = args.steps
    torch.cuda.synchronize()
    c0 = _lib.launch_count()
    runner.step(0)                                            # count the kernels of ONE step (outside the timed region)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - c0
    gpu_launches = timed_steps * launches_per_step
    value = timed_steps * B_TRAIN * T * world / (ms * 1e-3)
    final_loss = float(runner.loss[0].item())
    tc_status = int(_lib.load().b2h_tc_status())

    # ---------------- e2e: pinned host buffer -> ONE H2D copy -> step -> D2H loss, every step ----------------
    # runner.pipelined_steps: batch i+1 travels on a copy stream while step i computes (what a prefetching DataLoader
    # gives the reference loop); the loss of every step is read on the host inside the loop (one step behind the launch).
    from hand_pose_sl_b200.runner import pipelined_steps
    # Five back-to-back segments of 400 steps; the reported figure is the MEDIAN segment (a shared host's PCIe / memory
    # traffic moves single short segments by tens of percent), all five are listed.
    e2e_steps, e2e_segments = 400, 5
    h2d = int(staged[0].numel())
    for _ in pipelined_steps(runner, (staged[i % N_SLOTS] for i in range(10))):
        pass
    torch.cuda.synchronize()
    seg_dt = []
    n_p, loss_val = 0, float("nan")
    for _seg in range(e2e_segments):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        n_p = 0
        for loss_val in pipelined_steps(runner, (staged[i % N_SLOTS] for i in range(e2e_steps))):
            n_p += 1
        torch.cuda.synchronize()
        seg_dt.append(time.perf_counter() - t0)
    if world > 1:                                             # a segment takes as long as its slowest rank
        t = torch.tensor(seg_dt, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        seg_dt = [float(v) for v in t.tolist()]
    e2e_dt = sorted(seg_dt)[len(seg_dt) // 2]
    # sequential variant (copy, then step, then read) for reference
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(50):
        runner.load_staged(staged[i % N_SLOTS], slot=0)
        loss_val = float(runner.step(0).item())
    torch.cuda.synchronize()
    seq_dt = (time.perf_counter() - t0) / 50
    if world > 1:
        t = torch.tensor([seq_dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        seq_dt = float(t[0].item())
    e2e = {"value": n_p * B_TRAIN * T * world / e2e_dt, "unit": "frames/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": 4, "steps": n_p, "segments": e2e_segments,
           "segment_us_per_step": [round(v / max(n_p, 1) * 1e6, 2) for v in seg_dt], "statistic": "median segment",
           "api": "runner.pipelined_steps(runner, runner.host_stage(batch) buffers): per step ONE cudaMemcpyAsync of the pinned batch, "
                  "the step, and the loss read on the host (the kernel stores it into pinned host memory; read one step behind the launch)",
           "mode": "pipelined (double-buffered H2D on a copy stream)", "input_dtype": str(x_dt).replace("torch.", ""),
           "sequential_value": B_TRAIN * T * world / seq_dt, "us_per_step": e2e_dt / max(n_p, 1) * 1e6,
           "h2d_gbs": h2d / (e2e_dt / max(n_p, 1)) / 1e9}

    # ---------------- data-parallel parity, untimed (the driver's GPU test box has one GPU) ----------------
    dp_parity = None
    if world > 1:
        dp_parity = {"replicas_bit_identical_after_timed_run": bool(runner.replicas_identical()),
                     "peers_in_exchange_table": int(runner.peers_seen), "exchange": runner.exchange,
                     "multicast_push": bool(getattr(runner, "mc_ptr", 0))}
        try:
            dp_parity.update(dp_parity_check(b2h, synthetic, DataParallelTrainer, TrainStepRunner, dev, rank, world, train_prec,
                                             args.exchange, not args.no_multicast))
        except Exception as ex:   # noqa: BLE001
            dp_parity["error"] = f"{type(ex).__name__}: {ex}"[:300]
    try:
        runner.finish()
        status_ok = True
    except Exception as ex:   # noqa: BLE001
        status_ok = False
        sys.stderr.write(f"[bench] {ex}\n")

    line = {"metric": "body2hand_train_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / timed_steps, "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "f32" if train_prec.startswith("fp32") else "bf16", "data": "synthetic",
            "timed_steps": timed_steps, "timed_region_ms": ms,
            "config": {"workload": f"train step (fwd+mask+L1+bwd+Adam), batch {B_TRAIN}x{T} frames per GPU, C={C} (BASELINE config 3/4)",
                       "global_batch": B_TRAIN * world, "frames_per_window": T, "conv_channels": C,
                       "parallelism": f"dp{world}", "cuda_graph": graphed, "host_numa": host_numa,
                       "grad_exchange": (getattr(runner, "exchange", None) if world > 1 else None),
                       "timing": f"{args.steps} steps timed back to back after {max(args.warmup, chunk)} warm-up steps "
                                 f"of the same CUDA graph and one untimed {args.steps}-step pass that aligns the ranks",
                       "l2": f"{N_SLOTS} resident batches rotated ({N_SLOTS * (h2d) / 1e6:.0f} MB inputs + "
                             f"{_lib.workspace_bytes(B_TRAIN, T, 24, C, 0, _lib.PRECISIONS[train_prec]) / 1e6:.0f} MB gradient partials) > 126 MB L2"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(gpu_launches), "final_loss": final_loss,
            "tc_status": tc_status, "status_ok": status_ok}
    if world > 1:
        line["dp_parity"] = dp_parity
        line["comm_nranks"] = int(runner.peers_seen)

    if world > 1 and launches_per_step == 1:
        # per-GPU roofline of the one fused kernel (its in-kernel gradient exchange included); cpu_baseline is N=1 only
        k_ms = ms / timed_steps
        tfl = TRAIN_FLOP_PER_WINDOW * B_TRAIN / (k_ms * 1e-3) / 1e12
        line["roofline"] = {"bound": "tensor", "achieved": tfl, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": tfl / pk["tflops"],
                            "traffic": None, "kernel": "conv_tc_tile_kernel<train> (data-parallel tail)", "kernel_ms": k_ms,
                            "algorithmic_flop_per_launch": TRAIN_FLOP_PER_WINDOW * B_TRAIN,
                            "peak_source": pk["source"] + ", bf16 dense sustained",
                            "note": "per GPU: one cooperative launch per step per rank, peer-memory gradient exchange inside it"}
    if rank == 0 and world == 1:
        # ---------------- roofline of the dominant kernel (fused fwd+loss+bwd), timed alone ----------------
        lib = _lib.load()
        n_in, Cc, pe = model._geometry()

        def train_kernel_only(slot):
            _lib.check(lib.b2h_train_forward_backward(
                _lib.ptr(runner.x[slot]), runner._x_dt(), _lib.ptr(runner.target[slot]), None, _lib.ptr(runner.lengths[slot]),
                _lib.ptr(model._flat), _lib.ptr(runner.packed), None, None, None, B_TRAIN, T, n_in, Cc, pe, _lib.LOSS_L1,
                _lib.PRECISIONS[model.precision], None, _lib.ptr(runner.ws), runner.ws.numel(), _lib.stream_ptr(dev)))

        for i in range(10):
            train_kernel_only(i % N_SLOTS)
        torch.cuda.synchronize()
        kgraph = torch.cuda.CUDAGraph()                       # graph replay: device time, not Python launch rate
        with torch.cuda.graph(kgraph):
            for i in range(N_SLOTS):
                train_kernel_only(i)
        kgraph.replay()
        torch.cuda.synchronize()
        greps = 5
        reps = greps * N_SLOTS
        ev0.record()
        for _ in range(greps):
            kgraph.replay()
        ev1.record()
        torch.cuda.synchronize()
        k_only_ms = ev0.elapsed_time(ev1) / reps            # forward+loss+backward kernel without the fused tail
        fused = launches_per_step == 1                      # bf16 mode: the whole step IS one kernel launch
        k_ms = (ms / timed_steps) if fused else k_only_ms
        tfl = TRAIN_FLOP_PER_WINDOW * B_TRAIN / (k_ms * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.isfile(tpath):
            traffic = json.load(open(tpath)).get("train_kernel_dram_bytes_per_launch")
        line["roofline"] = {"bound": "tensor", "achieved": tfl, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": tfl / pk["tflops"],
                            "traffic": traffic, "kernel": "conv_fp32_kernel<train>" if train_prec == "fp32-ffma" else "conv_tc_tile_kernel<train>",
                            "kernel_ms": k_ms, "kernel_ms_fwd_bwd_only": k_only_ms, "algorithmic_flop_per_launch": TRAIN_FLOP_PER_WINDOW * B_TRAIN,
                            "peak_source": pk["source"] + ", bf16 dense sustained",
                            "note": "bf16 mode: one cooperative launch per step (fwd+loss+bwd, grid barrier, reduction, Adam), timed over the graph-replayed steps (inter-kernel gaps included); kernel_ms_fwd_bwd_only = the same kernel without its reduction/Adam tail; per-launch device times are in profiles/"}

        def time_train(prec, Bx, Tx, Cx=C, slots=8, reps=6):
            """graph-replayed train steps of another precision / shape (same API, same step definition)"""
            torch.manual_seed(0)
            mm = b2h.ConvModel(Cx, "ReLU", False, precision=prec).to(dev)
            oo = b2h.FusedAdam(mm.parameters(), lr=LR)
            rr = TrainStepRunner(mm, oo, Bx, Tx, "L1", n_slots=slots)
            for s_ in range(slots):
                rr.load(synthetic.model_batch(Bx, Tx, seed=500 + s_), slot=s_, non_blocking=False)
            rr.capture(slots)
            rr.replay(); rr.replay()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                rr.replay()
            ev1.record()
            torch.cuda.synchronize()
            rr.finish()
            t_ms = ev0.elapsed_time(ev1) / (reps * slots)
            sm = 24 * Cx + 2 * Cx * Cx + 42 * Cx
            flop = 2 * (5 * Tx - 6) * (3 * sm - 24 * Cx) * Bx
            return {"value": Bx * Tx / (t_ms * 1e-3), "unit": "frames/s", "ms_per_step": t_ms, "dtype": "f32" if prec.startswith("fp32") else "bf16",
                    "workload": f"train step, batch {Bx}x{Tx}, C={Cx}, CUDA graph", "final_loss": float(rr.loss[0].item()),
                    "kernel": {1: "ffma", 2: "tcgen05 tile" + (" (bf16 high/low operand pairs, 3 MMAs per product)" if prec == "fp32" else ""),
                               5: "tcgen05 wide (fwd+criterion / dgrad chain / split-K wgrad)"}.get(int(lib.b2h_kernel_choice(Tx, 24, Cx, 0, _lib.PRECISIONS[prec], 1)), "?"),
                    "roofline": {"bound": "tensor", "achieved": flop / (t_ms * 1e-3) / 1e12, "peak": pk["tflops"], "unit": "TFLOP/s",
                                 "frac": flop / (t_ms * 1e-3) / 1e12 / pk["tflops"]}}

        def time_fwd(prec, Bx, Tx, Cx=C, slots=8, reps=6, x_dtype=None):
            torch.manual_seed(0)
            mm = b2h.ConvModel(Cx, "ReLU", False, precision=prec).to(dev)
            xd = x_dtype or (torch.bfloat16 if prec == "bf16" else torch.float32)
            ff = ForwardRunner(mm, Bx, Tx, n_slots=slots, x_dtype=xd)
            for s_ in range(slots):
                ff.x[s_].copy_(synthetic.model_batch(Bx, Tx, seed=600 + s_)["input_kp"])
            ff.capture(slots)
            ff.graph.replay(); ff.graph.replay()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                ff.graph.replay()
            ev1.record()
            torch.cuda.synchronize()
            t_ms = ev0.elapsed_time(ev1) / (reps * slots)
            sm = 24 * Cx + 2 * Cx * Cx + 42 * Cx
            flop = 2 * (5 * Tx - 6) * sm * Bx
            return {"value": Bx * Tx / (t_ms * 1e-3), "unit": "frames/s", "ms_per_batch": t_ms, "dtype": "f32" if prec.startswith("fp32") else "bf16",
                    "workload": f"forward, batch {Bx}x{Tx}, C={Cx}, CUDA graph",
                    "roofline": {"bound": "tensor", "achieved": flop / (t_ms * 1e-3) / 1e12, "peak": pk["tflops"], "unit": "TFLOP/s",
                                 "frac": flop / (t_ms * 1e-3) / 1e12 / pk["tflops"]}}

        if not args.skip_extras:
            # ---------------- the same configs in fp32 mode (the reference's own precision, 1e-4 parity), the reference's
            # default shape (run.py:28,43: batch 128, 200-frame crops) and BASELINE config 1 (one 64-frame window) ----------------
            for key, fn in (("train_fp32", lambda: time_train("fp32", B_TRAIN, T)),
                            ("fwd_fp32", lambda: time_fwd("fp32", B_FWD, T)),
                            ("train_fp32_ffma", lambda: time_train("fp32-ffma", B_TRAIN, T)),
                            ("fwd_fp32_ffma", lambda: time_fwd("fp32-ffma", B_FWD, T)),
                            ("train_wide", lambda: time_train("bf16", B_TRAIN, T, Cx=256, slots=4, reps=5)),
                            ("train_wide_b444", lambda: time_train("bf16", 444, T, Cx=256, slots=2, reps=5)),     # 148 tiles: one per SM
                            ("train_wide_b888", lambda: time_train("bf16", 888, T, Cx=256, slots=2, reps=5)),
                            ("train_wide_c128", lambda: time_train("bf16", B_TRAIN, T, Cx=128, slots=4, reps=5)),
                            ("train_c64", lambda: time_train("bf16", B_TRAIN, T, Cx=64, slots=4, reps=5)),
                            ("train_ref_default_shape", lambda: time_train(train_prec, 128, 200)),
                            ("train_ref_default_shape_fp32", lambda: time_train("fp32", 128, 200)),
                            ("fwd_config1_latency", lambda: time_fwd(fwd_prec, 1, T, slots=4, reps=50)),
                            ("fwd_config1_latency_fp32", lambda: time_fwd("fp32", 1, T, slots=4, reps=50))):
                try:
                    line[key] = fn()
                except Exception as ex:   # noqa: BLE001
                    line[key] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        if not args.skip_extras:
            # ---------------- config 2: forward, batch 512 x 64, bf16 tensor-core path ----------------
            torch.manual_seed(0)
            fmodel = b2h.ConvModel(C, "ReLU", False, precision=fwd_prec).to(dev)
            fr = ForwardRunner(fmodel, B_FWD, T, n_slots=N_SLOTS, x_dtype=torch.bfloat16 if fwd_prec == "bf16" else torch.float32)
            for s in range(N_SLOTS):
                fr.x[s].copy_(synthetic.model_batch(B_FWD, T, seed=99 + s)["input_kp"])
            fr.capture(N_SLOTS)
            for _ in range(3):
                fr.graph.replay()
            torch.cuda.synchronize()
            freps = 10
            ev0.record()
            for _ in range(freps):
                fr.graph.replay()
            ev1.record()
            torch.cuda.synchronize()
            f_ms = ev0.elapsed_time(ev1) / (freps * N_SLOTS)
            f_tfl = FWD_FLOP_PER_WINDOW * B_FWD / (f_ms * 1e-3) / 1e12
            in_b = 2 if fwd_prec == "bf16" else 4
            f_bytes = B_FWD * T * (24 * in_b + 42 * 4)
            line["fwd"] = {"metric": "body2hand_forward_frames_per_sec", "value": B_FWD * T / (f_ms * 1e-3), "unit": "frames/s",
                           "ms_per_batch": f_ms, "dtype": fwd_prec, "workload": f"forward, batch {B_FWD}x{T} (BASELINE config 2), CUDA graph",
                           "roofline": {"bound": "tensor", "achieved": f_tfl, "peak": pk["tflops"], "unit": "TFLOP/s",
                                        "frac": f_tfl / pk["tflops"], "hbm_gbs": f_bytes / (f_ms * 1e-3) / 1e9,
                                        "hbm_frac": f_bytes / (f_ms * 1e-3) / 1e9 / pk["hbm_gbs"]},
                           "tc_status": int(lib.b2h_tc_status())}
            # ---------------- wide variant (SURVEY 8d: C = 256 puts the convs on the tensor-pipe roofline) ----------------
            if fwd_prec == "bf16":
                CW = 256
                sw = 24 * CW + 2 * CW * CW + 42 * CW
                wide = {}
                for (bw, tw) in ((1776, 64), (1184, 126)):       # 4 tiles of 256 rows per SM: 3 x 64-frame / 2 x 126-frame windows per tile
                    torch.manual_seed(0)
                    wm = b2h.ConvModel(CW, "ReLU", False, precision="bf16").to(dev)
                    wr = ForwardRunner(wm, bw, tw, n_slots=4, x_dtype=torch.bfloat16)
                    for s in range(4):
                        wr.x[s].copy_(synthetic.model_batch(bw, tw, seed=300 + s)["input_kp"])
                    wr.capture(8)
                    for _ in range(3):
                        wr.graph.replay()
                    torch.cuda.synchronize()
                    ev0.record()
                    for _ in range(5):
                        wr.graph.replay()
                    ev1.record()
                    torch.cuda.synchronize()
                    w_ms = ev0.elapsed_time(ev1) / 40
                    w_tfl = 2 * (5 * tw - 6) * sw * bw / (w_ms * 1e-3) / 1e12
                    w_traffic = None
                    if (bw, tw) == (1184, 126) and os.path.isfile(tpath):
                        w_traffic = json.load(open(tpath)).get("wide_fwd_dram_bytes_per_launch")
                    wide[f"{bw}x{tw}"] = {"value": bw * tw / (w_ms * 1e-3), "unit": "frames/s", "ms_per_batch": w_ms,
                                          "roofline": {"bound": "tensor", "achieved": w_tfl, "peak": pk["tflops"], "unit": "TFLOP/s",
                                                       "frac": w_tfl / pk["tflops"], "traffic": w_traffic}}
                    del wr, wm
                line["fwd_wide"] = {"metric": "body2hand_forward_frames_per_sec", "dtype": "bf16", "conv_channels": CW,
                                    "workload": "forward, conv_channels=256 (streamed-weight tcgen05 kernel), bf16 inputs, CUDA graph of 8 launches over 4 resident batches",
                                    "batches": wide, "tc_status": int(lib.b2h_tc_status())}
            # ---------------- K0 preprocessing: 2 h of 30 fps frames ----------------
            F = 216000
            pose, lh, rh = synthetic.synthetic_clip(F, seed=1234)
            tp, tl, tr = (torch.from_numpy(a).to(dev) for a in (pose, lh, rh))
            pre = b2h.PreprocessRightHand()
            starts = torch.zeros(1, dtype=torch.int64, device=dev)
            pout = pre(tp, tl, tr, starts, F)
            for _ in range(3):
                pre(tp, tl, tr, starts, F, out=pout)
            torch.cuda.synchronize()
            pgraph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(pgraph):
                for _ in range(4):
                    pre(tp, tl, tr, starts, F, out=pout)
            pgraph.replay()
            torch.cuda.synchronize()
            preps = 20
            ev0.record()
            for _ in range(preps // 4):
                pgraph.replay()
            ev1.record()
            torch.cuda.synchronize()
            p_ms = ev0.elapsed_time(ev1) / preps
            gbs = F * PRE_BYTES_PER_FRAME / (p_ms * 1e-3) / 1e9
            ptraffic = None
            if os.path.isfile(tpath):
                pf = json.load(open(tpath)).get("preprocess_dram_bytes_per_frame")
                ptraffic = pf * F if pf else None
            line["preprocess"] = {"metric": "body2hand_preprocess_frames_per_sec", "value": F / (p_ms * 1e-3), "unit": "frames/s",
                                  "ms_per_launch": p_ms, "workload": f"{F} frames (2 h at 30 fps), full reference item (1452 B/frame)",
                                  "roofline": {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                               "frac": gbs / pk["hbm_gbs"], "traffic": ptraffic,
                                               "note": "CUDA-graph replay, outputs reused; 314 MB moved per launch > 126 MB L2"}}
            # ---------------- K0, packed H5 rows (TextPoseH5Dataset.array2item): same kernel, 150-float rows ----------------
            try:
                rows = torch.randn(F, 150, device=dev) * 300 + 600
                rows[:, 100:] = torch.rand(F, 50, device=dev)
                h5o = pre.from_h5_rows(rows, starts, F)
                torch.cuda.synchronize()
                hgraph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(hgraph):
                    for _ in range(4):
                        h5o = pre.from_h5_rows(rows, starts, F)
                hgraph.replay()
                torch.cuda.synchronize()
                ev0.record()
                for _ in range(preps // 4):
                    hgraph.replay()
                ev1.record()
                torch.cuda.synchronize()
                h_ms = ev0.elapsed_time(ev1) / preps
                h_gbs = F * 1200 / (h_ms * 1e-3) / 1e9
                line["preprocess_h5"] = {"metric": "body2hand_preprocess_frames_per_sec", "value": F / (h_ms * 1e-3), "unit": "frames/s",
                                         "ms_per_launch": h_ms, "workload": f"{F} packed H5 rows (600 B read + 600 B written per frame)",
                                         "roofline": {"bound": "hbm", "achieved": h_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                                      "frac": h_gbs / pk["hbm_gbs"], "traffic": None}}
                del rows, h5o, hgraph
            except Exception as ex:   # noqa: BLE001
                line["preprocess_h5"] = {"error": f"{type(ex).__name__}: {ex}"[:200]}
        if not args.skip_extras:
            # ---------------- config 5: streaming K0 -> K1 over 1 h of frames (stride 64 and 16) ----------------
            # K0 runs ONCE per unique frame and writes only what the net reads (a (F,12,2) bf16 stream); the forward reads
            # the sliding windows as views of that stream (crop + pad rule on the fly): overlapping windows are never
            # materialised.  "materialised" = the round-1 pipeline (K0 writes every window's full item) for comparison.
            Fs = 108000
            sp_, sl_, sr_ = (t_[:Fs].contiguous() for t_ in (tp, tl, tr))
            line["stream"] = {"workload": f"{Fs} frames (1 h at 30 fps): K0 per unique frame -> bf16 frame stream -> forward over "
                                          f"64-frame window views (x1280 de-normalise fused), CUDA graph", "dtype": fwd_prec}
            for stride in (64, 16):
                st_np = b2h.sliding_window_starts(Fs - T + 1, T, stride)
                st_ = torch.from_numpy(st_np).to(dev)
                Wn = st_.numel()
                entry = {"windows": Wn}
                if fwd_prec == "bf16":
                    pre_v = b2h.PreprocessRightHand()
                    stream_buf = pre_v.frame_stream(sp_, sl_, sr_)
                    yv = fmodel.predict_windows(stream_buf, st_, T, denormalize=1280.0)
                    torch.cuda.synchronize()
                    sg = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(sg):
                        for _ in range(4):
                            pre_v.frame_stream(sp_, sl_, sr_, out=stream_buf)
                            fmodel.predict_windows(stream_buf, st_, T, denormalize=1280.0, out=yv)
                    sg.replay(); torch.cuda.synchronize()
                    ev0.record()
                    for _ in range(5):
                        sg.replay()
                    ev1.record()
                    torch.cuda.synchronize()
                    s_ms = ev0.elapsed_time(ev1) / 20
                    entry.update({"ms": s_ms, "unique_frames_per_sec": Fs / (s_ms * 1e-3), "window_frames_per_sec": Wn * T / (s_ms * 1e-3),
                                  "path": "window views of the per-frame stream (no re-materialisation)"})
                    del sg
                pre_s = b2h.PreprocessRightHand(with_left_hand=False, emit_bf16=(fwd_prec == "bf16"))
                so = pre_s(sp_, sl_, sr_, st_, T)
                xin = so["input_kp_bf16"] if fwd_prec == "bf16" else so["input_kp"]
                frs = ForwardRunner(fmodel, Wn, T, n_slots=1, x_dtype=xin.dtype, out_scale=1280.0)
                frs.x = xin.view(1, Wn, T, 12, 2)              # the net reads K0's output in place (no copy)
                pre_s(sp_, sl_, sr_, st_, T, out=so); frs.run(0)
                torch.cuda.synchronize()
                sg = torch.cuda.CUDAGraph()
                with torch.cuda.graph(sg):
                    for _ in range(4):
                        pre_s(sp_, sl_, sr_, st_, T, out=so)
                        frs.run(0)
                sg.replay(); torch.cuda.synchronize()
                ev0.record()
                for _ in range(5):
                    sg.replay()
                ev1.record()
                torch.cuda.synchronize()
                m_ms = ev0.elapsed_time(ev1) / 20
                entry["materialised"] = {"ms": m_ms, "unique_frames_per_sec": Fs / (m_ms * 1e-3)}
                if "ms" not in entry:
                    entry.update({"ms": m_ms, "unique_frames_per_sec": Fs / (m_ms * 1e-3), "window_frames_per_sec": Wn * T / (m_ms * 1e-3),
                                  "path": "materialised windows"})
                line["stream"][f"stride{stride}"] = entry
                del sg, frs, so
            # ---- the same pipeline over 8 h of frames (SURVEY 8d config 5): window views only; the clip is the 2 h clip x 4 ----
            if fwd_prec == "bf16":
                try:
                    F8 = 4 * F
                    lp_, ll_, lr_ = (t_.repeat(4, 1, 1) for t_ in (tp, tl, tr))
                    pre_v = b2h.PreprocessRightHand()
                    stream8 = pre_v.frame_stream(lp_, ll_, lr_)
                    long_run = {"frames": F8}
                    for stride in (64, 16):
                        st_ = torch.from_numpy(b2h.sliding_window_starts(F8 - T + 1, T, stride)).to(dev)
                        Wn = st_.numel()
                        yv = fmodel.predict_windows(stream8, st_, T, denormalize=1280.0)
                        torch.cuda.synchronize()
                        sg = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(sg):
                            for _ in range(2):
                                pre_v.frame_stream(lp_, ll_, lr_, out=stream8)
                                fmodel.predict_windows(stream8, st_, T, denormalize=1280.0, out=yv)
                        sg.replay(); torch.cuda.synchronize()
                        ev0.record()
                        for _ in range(3):
                            sg.replay()
                        ev1.record()
                        torch.cuda.synchronize()
                        l_ms = ev0.elapsed_time(ev1) / 6
                        long_run[f"stride{stride}"] = {"windows": Wn, "ms": l_ms, "unique_frames_per_sec": F8 / (l_ms * 1e-3),
                                                       "window_frames_per_sec": Wn * T / (l_ms * 1e-3)}
                        del sg, yv, st_
                    line["stream"]["clip_8h"] = long_run
                    del lp_, ll_, lr_, stream8
                except Exception as ex:   # noqa: BLE001
                    line["stream"]["clip_8h"] = {"error": f"{type(ex).__name__}: {ex}"[:200]}
        # ---------------- CPU baseline (reference path on this box's host cores) ----------------
        line["cpu_baseline"], _, _ = cpu_reference_arm(200, 2, budget_s=15.0)
        if not args.skip_extras:
            # ---------------- launch-latency floor (SURVEY 8d): 40 dependent one-block kernels per graph replay ----------------
            # Last on purpose and fully guarded: nothing measured above can be affected by it.
            try:
                tiny = torch.zeros((1, 1, 21, 2), dtype=torch.float32, device=dev)
                tlen = torch.ones(1, dtype=torch.int32, device=dev)
                from hand_pose_sl_b200 import _lib as _l

                def _tiny():
                    _l.check(lib.b2h_mask_output(_l.ptr(tiny), _l.ptr(tlen), 1, 1, 42, _l.stream_ptr(dev)))
                _tiny()
                torch.cuda.synchronize()
                fg = torch.cuda.CUDAGraph()
                with torch.cuda.graph(fg):
                    for _ in range(40):
                        _tiny()
                fg.replay()
                torch.cuda.synchronize()
                ev0.record()
                for _ in range(10):
                    fg.replay()
                ev1.record()
                torch.cuda.synchronize()
                line["launch_floor_us"] = ev0.elapsed_time(ev1) * 1e3 / 400
            except Exception as e:   # noqa: BLE001
                line["launch_floor_us"] = None
                line["launch_floor_error"] = str(e)[:200]

    sys.stdout.flush()
    try:                                   # NCCL's banner sits in the C stdio buffer: push it to the redirected fd first
        import ctypes
        ctypes.CDLL(None).fflush(None)
    except Exception:
        pass
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tearing the NCCL communicator down while a captured CUDA graph still holds its kernels hangs in
        # destroy_process_group (seen on B200, torch 2.11 / NCCL 2.28): synchronise, then leave without the teardown.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
