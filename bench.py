#!/usr/bin/env python
"""Headline benchmark: frames/s of one BLSTM-CTC training step (BASELINE.json config 2:
5x512 BLSTM, 80-d input, T=1000, B=64 per GPU, 28 chars + blank), data-parallel over N GPUs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = forward (5 BLSTM layers + output FC) + CTC loss/grad + backward (BPTT + weight
gradients) + per-tensor clip_by_norm + gradient all-reduce (N>1) + RMSProp update.
`value`  : frames/s with the batch already resident in HBM (device-timed, CUDA events).
`e2e`    : the same step through the public model API with HOST (pinned) buffers: every step's H2D
           copy of its batch (PinnedPrefetcher: side stream, issued one step ahead) and the D2H read of
           its loss (asynchronous, consumed one step later) are inside the timed region.
`--impl reference` times the CPU restatement of the reference's TF-1.x step
(oracle/model.py, torch-CPU, all host threads) on a bounded sample -- the real TF1 CPU
path cannot run here (TensorFlow is not installable; BASELINE.md #2).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(input_size=80, num_units=512, num_layers=5, num_classes=28, T=1000, B=64,
           label_min=150, label_max=250, optimizer="rmsprop", lr=1e-3, clip=5.0,
           keep_prob=float(os.environ.get("B2_BENCH_KEEP_PROB", "0.8")))   # dropout 0.2: blstm_ctc_960h_char.yml:34
# SURVEY 8(d): forward MAC count of the gate GEMMs, x3 for training
FWD_FLOP_PER_FRAME = 2 * 2 * (80 + 512) * 2048 + 4 * 2 * 2 * (1024 + 512) * 2048   # 55.18 M
# weak: 64 utterances per GPU (default, the driver's convention); strong: the reference's own semantics --
# ONE global batch of 64 np.array_split over the ranks (utils/dataset/ctc.py:171-177)
SCALING = os.environ.get("B2_BENCH_SCALING", "weak")
# CPU arm: one step = full model on CPU_B utterances x CPU_T frames, fixed thread count
CPU_B, CPU_T = int(os.environ.get("B2_BENCH_CPU_B", "8")), int(os.environ.get("B2_BENCH_CPU_T", "1000"))
CPU_THREADS = int(os.environ.get("B2_BENCH_CPU_THREADS", "32"))


def make_batch(seed, B, T, D, C, lmin, lmax):
    rng = np.random.RandomState(seed)
    x = rng.randn(B, T, D).astype(np.float32)
    seq = np.full(B, T, np.int32)
    labels = [list(rng.randint(0, C, size=int(rng.randint(lmin, lmax + 1)))) for _ in range(B)]
    return x, seq, labels


class ClockSampler(object):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
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
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_baseline(B_s, T_s, threads=None, steps=1):
    """CPU restatement of the same train step on a bounded sample (B_s utterances x T_s frames,
    full 5x512 model).  Returns frames/s."""
    import torch
    from oracle import model as omodel
    from oracle import lstm as olstm
    if threads:
        torch.set_num_threads(threads)
    rng = np.random.RandomState(0)
    layers = olstm.init_blstm_params(CFG["input_size"], CFG["num_units"], CFG["num_layers"], seed=0)
    vs = {}
    for i, l in enumerate(layers, 1):
        for d in ("fw", "bw"):
            for k, v in l[d].items():
                vs["blstm_hidden%d/%s/lstm_cell/%s" % (i, d, k)] = v
    C = CFG["num_classes"] + 1
    vs["output/weights"] = (rng.randn(2 * CFG["num_units"], C) * 0.1).astype(np.float32)
    vs["output/biases"] = np.zeros(C, np.float32)
    tr = omodel.OracleTrainer(vs, CFG["num_layers"], optimizer=CFG["optimizer"], learning_rate=CFG["lr"],
                              clip_grad_norm=CFG["clip"], dtype=torch.float32)
    lmax = max(2, int(CFG["label_max"] * T_s / CFG["T"]))
    lmin = max(1, int(CFG["label_min"] * T_s / CFG["T"]))
    x, seq, labels = make_batch(1, B_s, T_s, CFG["input_size"], CFG["num_classes"], lmin, lmax)
    t0 = time.time()
    for _ in range(steps):
        tr.step(x, seq, labels)
    dt = (time.time() - t0) / steps
    return B_s * T_s / dt, dt


def cpu_arm_record(v, dt, threads, nsteps):
    sample = ("one full train step (fwd + CTC + bwd + clip + rmsprop) of the config-2 model (5x512 BLSTM, 80-d, "
              "C=29) on B=%d utterances x T=%d frames = %d frames, %.1f s; frames/s is per frame, so the B=64 "
              "figure is this value (per-step work is linear in B)" % (CPU_B, CPU_T, CPU_B * CPU_T, dt))
    return {"value": v, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample,
            "cpu_model": cpu_model_name(), "host_cpus": os.cpu_count(), "timed_steps": nsteps,
            "note": "torch-CPU restatement of the TF-1.x step (oracle/model.py, fp32, %d intra-op threads); "
                    "TensorFlow itself is not installable here" % threads}


DUMP_SAMPLE = 1 << 20      # elements of the flat parameter / gradient buffers written by --dump-outputs


def restore_initial_state(model, params0):
    """Parameters as constructed and optimizer slots as created, so that the step that follows starts from the
    same state in every run.  Without it the last step's inputs would be the product of every earlier step, and
    those carry the run-to-run rounding of the atomic gradient reductions (measured on a B200 at 1000 W: 1e-4
    relative in the loss after a dozen steps, near 10 % after fifty)."""
    from tensorflow_end2end_speech_recognition_b200.models.model_base import OPTIMIZER_CLS_NAMES
    model.flat_params.copy_(params0)
    model._params_version += 1
    opt = model.optimizer
    if opt.state0 is not None:
        opt.state0.fill_(OPTIMIZER_CLS_NAMES[opt.name][2])
    if opt.state1 is not None:
        opt.state1.zero_()
    opt.global_step = 0


def dump_outputs(out_dir, model, loss, logits):
    """What a caller of the timed step receives after its last step: the mean CTC loss, the per-utterance
    losses, the logits [T,B,C], and the parameters the optimizer updated (with the clipped gradients it
    applied).  The flat buffers (over 100 MB each) are sampled at fixed indices (seed 0, sorted), so that two
    builds write arrays that compare element for element.  About 16 MB in all."""
    import torch
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    n = model.flat_params.numel()
    idx = np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_SAMPLE), replace=False))
    idx_dev = torch.from_numpy(idx).to(model.flat_params.device)
    arrays = {"loss": loss.detach().reshape(1).double(),
              "ctc_losses": model.ctc_losses.detach().float(),
              "logits": logits.detach().float(),
              "params_sample": model.flat_params[idx_dev].float(),
              "grads_sample": model.flat_grads[idx_dev].float()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_reference(args):
    """--impl reference: CPU port of the reference step, rank 0 only.  One step = the bounded sample
    CPU_B x CPU_T (T stays 1000); at ~1 minute per step the arm times min(K, 2) steps after min(W, 1)
    warm-up so that the whole run ends within a few minutes, and says so in "steps"/"warmup"."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, CPU_THREADS)
    k_eff, w_eff = max(1, min(args.steps, 2)), min(args.warmup, 1)
    vals = []
    for i in range(w_eff + k_eff):
        v, dt = cpu_baseline(CPU_B, CPU_T, threads=threads, steps=1)
        if i >= w_eff:
            vals.append((v, dt))
    v = float(np.mean([a for a, _ in vals]))
    dt = float(np.mean([b for _, b in vals]))
    out = {"impl": "reference", "metric": "frames/sec BLSTM-CTC train", "value": v, "unit": "frames/s",
           "n_gpus": args.gpus, "steps": k_eff, "warmup": w_eff, "ms_per_step": dt * 1e3,
           "higher_is_better": True, "scaling": SCALING, "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": "BASELINE configs[1]: LibriSpeech-shape char CTC, 5x512 BLSTM, 80-d, "
                                  "T=1000, B=64 (CPU arm: bounded sample B=%d x T=%d, see cpu_baseline.sample)"
                                  % (CPU_B, CPU_T)},
           "cpu_baseline": cpu_arm_record(v, dt, threads, k_eff),
           "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0): loss, ctc_losses, "
                         "logits, and a fixed seeded sample of the updated parameters and of the gradients; that "
                         "step starts from the seeded initial parameters and optimizer state, restored inside the "
                         "timed region (one parameter-buffer copy and one optimizer-slot fill)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from tensorflow_end2end_speech_recognition_b200 import _lib, ops
    from tensorflow_end2end_speech_recognition_b200.models.ctc.ctc import CTC

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    B, T, D = CFG["B"], CFG["T"], CFG["input_size"]
    if SCALING == "strong":
        # the reference's semantics: one global batch of 64, np.array_split over the towers
        from tensorflow_end2end_speech_recognition_b200.utils.io.inputs.pipeline import shard_bounds
        lo, hi = shard_bounds(CFG["B"], world)[rank]
        B = hi - lo
    model = CTC(encoder_type="blstm", input_size=D, num_units=CFG["num_units"],
                num_layers=CFG["num_layers"], num_classes=CFG["num_classes"],
                lstm_impl="LSTMBlockCell", use_peephole=True, parameter_init=0.1,
                clip_grad_norm=CFG["clip"], precision=args.precision, device=dev, seed=1)
    comm, comm_kind = None, "none"
    if world > 1:
        comm_kind = "torch.distributed all_reduce (one call after BPTT)"
        if os.environ.get("B2_BENCH_COMM", "c_abi") == "c_abi":
            try:     # NCCL bound from the C ABI (b2_allreduce_mean), per-layer buckets overlapped with BPTT
                from tensorflow_end2end_speech_recognition_b200.utils.training.multi_gpu import NcclComm
                comm = NcclComm(rank, world, device=dev)
                comm_kind = "b2_allreduce_mean (NCCL from the C ABI), per-layer buckets overlapped with BPTT"
            except Exception as e:          # keep the run alive on the torch path, and say so
                comm, comm_kind = None, "torch.distributed all_reduce (C-ABI communicator failed: %s)" % (e,)
    model.set_data_parallel(world, comm=comm)
    # the seeded initial parameters, restored before the last timed step of a --dump-outputs run
    params0 = model.flat_params.clone() if args.dump_outputs else None
    # weak scaling: every rank gets its own 64-utterance shard (np.array_split of a 64*N batch,
    # utils/dataset/ctc.py:171-177); strong scaling: its slice of the one 64-utterance batch
    x, seq, labels = make_batch(1234 + rank, B, T, D, CFG["num_classes"], CFG["label_min"], CFG["label_max"])
    x_host = torch.from_numpy(x).pin_memory()
    seq_host = torch.from_numpy(seq).pin_memory()
    x_dev, seq_dev = x_host.to(dev), seq_host.to(dev)

    last = {}

    def step(xin, sin):
        loss, logits = model.compute_loss(xin, labels, sin, keep_prob=CFG["keep_prob"])
        model.train(loss, CFG["optimizer"], CFG["lr"])
        last["outputs"] = (loss, logits)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # e2e: every step copies ITS batch host -> device (pinned, on the prefetcher's side stream, issued one step
    # ahead so that it overlaps the previous step) and reads ITS loss device -> host (asynchronous copy into
    # pinned memory, consumed one step later so the host never drains the launch queue); both transfers of
    # every step lie inside the timed region, the final loss is read before the closing barrier.
    from tensorflow_end2end_speech_recognition_b200.utils.io.inputs.pipeline import PinnedPrefetcher
    pre = PinnedPrefetcher(dev)
    loss_host = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]
    loss_ev = [None, None]
    state = {"i": 0}
    pre.put(x_host, seq_host)

    def e2e_step():
        i = state["i"]
        xin, sin = pre.get()                   # this step's batch (H2D issued during the previous step)
        loss = step(xin, sin)
        pre.release()
        pre.put(x_host, seq_host)              # H2D of the next step's batch, overlapping this step
        k = i & 1
        loss_host[k].copy_(loss.detach().reshape(1), non_blocking=True)       # D2H of this step's result
        ev = torch.cuda.Event()
        ev.record()
        loss_ev[k] = ev
        if loss_ev[k ^ 1] is not None:         # consume the previous step's loss
            loss_ev[k ^ 1].synchronize()
            last["loss"] = float(loss_host[k ^ 1][0])
        state["i"] = i + 1

    def e2e_flush():
        k = (state["i"] - 1) & 1
        if loss_ev[k] is not None:
            loss_ev[k].synchronize()
            last["loss"] = float(loss_host[k][0])

    # warm up BOTH step flavours (allocator pools, module attributes, clocks) before timing
    for _ in range(max(args.warmup, 3)):
        step(x_dev, seq_dev)
    for _ in range(2):
        e2e_step()
    for _ in range(2):
        step(x_dev, seq_dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    try:
        l0 = lib.b2_launch_count()
        ms_dev = timed(lambda: step(x_dev, seq_dev), args.steps)
        launches = (lib.b2_launch_count() - l0) // args.steps

        last_i = state["i"] + args.steps - 1

        def e2e_loop_body():
            if params0 is not None and state["i"] == last_i:
                restore_initial_state(model, params0)
            e2e_step()
        ms_e2e = timed(e2e_loop_body, args.steps)
        e2e_flush()
    finally:
        clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, *last["outputs"])

    frames = (CFG["B"] if SCALING == "strong" else B * world) * T
    value = frames * args.steps / (ms_dev / 1e3)
    e2e = frames * args.steps / (ms_e2e / 1e3)
    ms_step = ms_dev / args.steps

    # ---- rooflines of the three kernel families, timed live with CUDA events (rank 0)
    roof = {}
    if rank == 0:
        peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
        try:
            pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            peaks.update({k: pk[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in pk})
            peaks["src"] = "measured"
        except Exception:
            pass

        def time_ms(fn, n=5):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        import ctypes as C
        TB, H = B * T, CFG["num_units"]
        A = torch.randn(TB, 2 * H, device=dev).bfloat16()
        W = torch.randn(8 * H, 2 * H, device=dev).bfloat16()
        Cm = torch.empty(TB, 8 * H, device=dev)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        t_gemm = time_ms(lambda: lib.b2_gemm_bf16(0, 0, TB, 8 * H, 2 * H, 1.0, C.c_void_p(A.data_ptr()), 2 * H,
                                                  C.c_void_p(W.data_ptr()), 2 * H, C.c_void_p(Cm.data_ptr()),
                                                  8 * H, C.c_void_p(0), 0, 0, st))
        fl = 2.0 * TB * 8 * H * 2 * H
        roof["blstm_gate_gemm"] = {"kernel": "gemm_tc_kernel<256> (time-batched gate GEMM, layers 2-5 forward)",
                                   "bound": "tensor", "achieved": fl / t_gemm / 1e9, "peak": peaks["bf16_tflops"],
                                   "unit": "TFLOP/s", "frac": fl / t_gemm / 1e9 / peaks["bf16_tflops"],
                                   "traffic": None, "ms": t_gemm, "peak_src": peaks["src"] + " burst"}
        del A, W, Cm
        # CTC at the bench shape
        Cc = CFG["num_classes"] + 1
        lg = torch.randn(T, B, Cc, device=dev)
        flat, offs, lmax = ops.pack_labels(labels)
        dflat, doffs = torch.tensor(flat, device=dev), torch.tensor(offs, device=dev)
        t_ctc = time_ms(lambda: ops.ctc_loss_grad(lg, dflat, doffs, seq_dev, lmax))
        # SURVEY 8(d): algorithmic bytes = 8*T*B*C (read logits, write grad) + 8*T*B*S alpha spill, S = 2*mean(L)+1
        s_mean = 2.0 * float(np.mean([len(l) for l in labels])) + 1.0
        by = 8.0 * T * B * Cc + 8.0 * T * B * s_mean
        roof["ctc_alpha_beta"] = {"kernel": "ctc_ab_team + ctc_softmax_rows + ctc_occ_rows + ctc_finalize", "bound": "hbm",
                                  "achieved": by / t_ctc / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                  "frac": by / t_ctc / 1e6 / peaks["hbm_gbs"], "traffic": None, "ms": t_ctc,
                                  "achieved_logits_only": 8.0 * T * B * Cc / t_ctc / 1e6,
                                  "note": "latency-bound at C=29 (T sequential lattice steps); algorithmic bytes = "
                                          "8*T*B*C + 8*T*B*S (S = 2*mean label length + 1, unpadded)",
                                  "peak_src": peaks["src"]}
        # the persistent recurrence kernels (dominant share of the step), timed with CUDA events
        # placed around their launches inside the library
        Hh = CFG["num_units"]
        prng = np.random.RandomState(0)
        Pl = {}
        for d in ("fw", "bw"):        # U(-0.1, 0.1) kernels / peepholes, zero bias (blstm.py:79-80)
            Pl[d] = {"kernel": torch.tensor(prng.uniform(-0.1, 0.1, (3 * Hh, 4 * Hh)).astype(np.float32), device=dev),
                     "bias": torch.zeros(4 * Hh, device=dev)}
            for k in ("w_i_diag", "w_f_diag", "w_o_diag"):
                Pl[d][k] = torch.tensor(prng.uniform(-0.1, 0.1, Hh).astype(np.float32), device=dev)
        Gl = {d: {k: torch.zeros_like(v) for k, v in Pl[d].items()} for d in Pl}
        xx = torch.randn(T, B, 2 * Hh, device=dev)
        dyy = torch.randn(T, B, 2 * Hh, device=dev)
        desc = ops.lstm_desc(T, B, 2 * Hh, Hh, precision=ops.PREC_BF16 if args.precision == "bf16" else ops.PREC_FP32)
        lib.b2_blstm_profile_enable(1)
        f_ms, b_ms = [], []
        for it in range(4):
            yy, _, res = ops.blstm_layer_forward(desc, xx, seq_dev, Pl["fw"], Pl["bw"])
            ops.blstm_layer_backward(desc, xx, seq_dev, Pl["fw"], Pl["bw"], dyy, res, Gl["fw"], Gl["bw"])
            ops.blstm_backward_join()
            torch.cuda.synchronize()
            fm, bm = C.c_float(0), C.c_float(0)
            if lib.b2_blstm_profile_last_ms(C.byref(fm), C.byref(bm)) == 0 and it > 0:
                f_ms.append(fm.value); b_ms.append(bm.value)
        lib.b2_blstm_profile_enable(0)
        del xx, dyy, yy, res
        if f_ms and min(f_ms) > 0:
            rec_fl = 2.0 * T * B * 2 * Hh * 4 * Hh            # h.Wh over T steps, both directions
            tf_, tb_ = float(np.median(f_ms)), float(np.median(b_ms))
            roof["blstm_recurrence_fwd"] = {
                "kernel": "lstm_rec_fwd_kernel<2,32> (persistent cluster/TMEM recurrence, one layer, T=1000)",
                "bound": "tensor", "achieved": rec_fl / tf_ / 1e9, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": rec_fl / tf_ / 1e9 / peaks["bf16_tflops"], "traffic": 2.84e9, "traffic_src": "static: ncu dram bytes "
                "read+write of one launch, profiles/prof_rec_fwd_r02_final_metrics.csv (not re-measured in this run)", "ms": tf_,
                "note": "latency-bound: 1000 dependent steps (tensor-pipe issue + DSMEM all-gather + gate math)",
                "peak_src": peaks["src"] + " burst"}
            roof["blstm_recurrence_bwd"] = {
                "kernel": "lstm_rec_bwd_kernel<2> (BPTT, one layer)", "bound": "tensor",
                "achieved": rec_fl / tb_ / 1e9, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": rec_fl / tb_ / 1e9 / peaks["bf16_tflops"], "traffic": 2.08e9, "traffic_src": "static: ncu dram bytes "
                "read+write of one launch, profiles/prof_rec_bwd_r02_final_metrics.csv (not re-measured in this run)", "ms": tb_,
                "note": "latency-bound (DSMEM reduce-scatter + gate math + tensor-pipe issue per step)",
                "peak_src": peaks["src"] + " burst"}
        # whole step against the tensor roofline (algorithmic gate-GEMM FLOPs / step time)
        step_fl = 3.0 * FWD_FLOP_PER_FRAME * B * T
        roof["step_blended"] = {"kernel": "whole training step (algorithmic gate-GEMM FLOPs / step time)",
                                "bound": "tensor", "achieved": step_fl / ms_step / 1e9,
                                "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                "frac": step_fl / ms_step / 1e9 / peaks["bf16_tflops_sustained"],
                                "traffic": None, "peak_src": peaks["src"] + " sustained"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = min(os.cpu_count() or 1, CPU_THREADS)
        # bounded: one step of the T=1000 sample at a quarter of the reference arm's batch
        v, dt = cpu_baseline(max(1, CPU_B // 4), CPU_T, threads=threads, steps=1)
        cpu = cpu_arm_record(v, dt, threads, 1)
        cpu["sample"] = cpu["sample"].replace("B=%d utterances" % CPU_B, "B=%d utterances" % max(1, CPU_B // 4)) \
            .replace("= %d frames" % (CPU_B * CPU_T), "= %d frames" % (max(1, CPU_B // 4) * CPU_T))

    if rank == 0:
        out = {"metric": "frames/sec BLSTM-CTC train", "value": value, "unit": "frames/s", "n_gpus": world,
               "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
               "higher_is_better": True, "scaling": SCALING, "vs_baseline": None, "dtype": args.precision,
               "data": "synthetic",
               "config": {"workload": "BASELINE configs[1]: LibriSpeech-shape char CTC, 5x512 BLSTM "
                                      "(LSTMBlockCell, peephole), 80-d input, T=1000, %s, "
                                      "28 chars + blank, labels 150-250, rmsprop lr 1e-3, clip_by_norm 5, "
                                      "dropout keep_prob %.2f" % (
                                          "B=64 per GPU" if SCALING != "strong" else
                                          "global B=64 array_split over the GPUs", CFG["keep_prob"]),
                          "global_batch": (CFG["B"] if SCALING == "strong" else B * world), "per_gpu_batch": B, "parallelism": "dp%d" % world,
                          "gradient_exchange": comm_kind,
                          "l2": "per-step working set (reserve + gate buffers, >8 GB) >> 126 MB L2, "
                                "no explicit flush"},
               "e2e": {"value": e2e, "unit": "frames/s", "ms_per_step": ms_e2e / args.steps,
                       "h2d_bytes_per_step": int(x_host.numel() * 4 + seq_host.numel() * 4 + sum(len(l) for l in labels) * 4 + (B + 1) * 4),
                       "d2h_bytes_per_step": 4, "loss": last.get("loss"),
                       "note": "per step: H2D of the step's batch from pinned memory on a side stream (issued one "
                               "step ahead, PinnedPrefetcher) + async D2H of the step's loss (host consumes it one "
                               "step later); both inside the timed region, overlapped with compute"},
               "gpu_launches": int(launches),
               "clocks": clocks,
               # dominant kernel by time share (profiles/README.md: recurrence 72 % of the step)
               "roofline": roof.get("blstm_recurrence_bwd") or roof.get("blstm_gate_gemm"),
               "rooflines": roof,
               "cpu_baseline": cpu}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
